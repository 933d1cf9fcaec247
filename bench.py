#!/usr/bin/env python
"""Benchmark of the predictor–corrector sampling hot path (BASELINE.json metric).

Metric: PC-sampler images/sec, NCSN++ cont. CIFAR-10, VE-SDE, 1000 steps
(``configs/ve/cifar10_ncsnpp_continuous.py`` with ``model.init_scale = 1``, random-init
weights, Gaussian-noise inputs).  A bench *step* is one PC iteration over one batch
(Langevin corrector + reverse-diffusion predictor = 2 network evaluations + both state
updates with in-kernel noise); a full sample is 1000 such steps, so

    images/s = n_gpus * batch / (1000 * seconds_per_step).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --gpus 1 --steps 2 --warmup 1     # CPU arm (oracle port)

One JSON line on stdout (rank 0).  `value` times the CUDA-graph replay loop with the state
resident in HBM; `e2e` goes through the public sampler plan with pinned host buffers
(H2D of the state and D2H of the result inside every timed step).
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

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

ALG_FLOP_PER_IMG_STEP = 43.58e9      # SURVEY.md §8(d): 2 evals x 21.788 GFLOP (2*MAC), measured on the reference
ALG_BYTES_PER_IMG_STEP = 153.9e6     # SURVEY.md §8(d): fp32 contraction operands only, everything else fused
N_SAMPLER_STEPS = 1000


def load_peaks():
  p = os.path.join(REPO, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    with open(p) as fh:
      d = json.load(fh)
    return dict(hbm_gbs=d['hbm_gbs'], bf16_tflops=d['bf16_tflops'], bf16_tflops_sustained=d['bf16_tflops_sustained'],
                source='measured (MEASURED_PEAKS.json)')
  return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
  """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

  def __init__(self, index):
    self.index, self.rows, self.proc = index, [], None

  def start(self):
    q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    try:
      self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                    '-lms', '200'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      threading.Thread(target=self._pump, daemon=True).start()
    except OSError:
      self.proc = None

  def _pump(self):
    for line in self.proc.stdout:
      self.rows.append([c.strip() for c in line.split(',')])

  def stop(self):
    if self.proc is None:
      return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
    self.proc.terminate()
    sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace('.', '').isdigit()]
    mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace('.', '').isdigit()]
    reasons = set()
    for r in self.rows:
      if len(r) >= 7:
        for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
          if v.lower().startswith('active'):
            reasons.add(name)
    return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                reasons=sorted(reasons), samples=len(sm))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
  """Write what the timed path returned in its last step as <out_dir>/<name>.npy (float64 stays float64, everything
  else is written as float32).  Above DUMP_LIMIT_BYTES in all, the same images (dim 0) of every array are kept, chosen
  by a fixed seed, so that two builds run with the same arguments can be compared array by array."""
  os.makedirs(out_dir, exist_ok=True)
  arrays = {k: v.detach().cpu() for k, v in arrays.items()}
  arrays = {k: v.double() if v.dtype == torch.float64 else v.float() for k, v in arrays.items()}
  n = arrays[next(iter(arrays))].shape[0]
  per_image = sum(v[0].numel() * v.element_size() for v in arrays.values())
  keep = min(n, DUMP_LIMIT_BYTES // per_image)
  if keep < n:
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    arrays = {k: v[idx] for k, v in arrays.items()}
  for k, v in arrays.items():
    np.save(os.path.join(out_dir, k + '.npy'), v.numpy())


SEPARATE_GROUPNORM_DEFAULT = True   # the plan bench.py measures by default = the package default (the faster one in the same-run A/B; both are in `variants`)


def headline_config():
  from score_sde_pytorch_b200 import configs
  cfg = configs.ve_cifar10_ncsnpp_continuous()
  cfg.model.init_scale = 1.0          # BASELINE.md §2: init_scale=0 zeroes every block's last conv
  return cfg


# ----------------------------------------------------------------------------------------------
# CPU arm: the UNMODIFIED reference (baseline/_ref, installed by tools/install_ref.sh) on the host cores
# ----------------------------------------------------------------------------------------------
REF_DIR = os.path.join(REPO, 'baseline', '_ref')
REF_EXT_DIR = os.path.join(REPO, 'baseline', '_ref_ext')


def physical_cores():
  """Physical cores this process may run on (hyper-thread siblings counted once), capped by the affinity mask."""
  try:
    allowed = sorted(os.sched_getaffinity(0))
  except AttributeError:
    allowed = list(range(os.cpu_count() or 1))
  seen, cores = set(), []
  for cpu in allowed:
    try:
      with open(f'/sys/devices/system/cpu/cpu{cpu}/topology/core_id') as fh:
        core = fh.read().strip()
      with open(f'/sys/devices/system/cpu/cpu{cpu}/topology/physical_package_id') as fh:
        pkg = fh.read().strip()
      key = (pkg, core)
    except OSError:
      key = ('?', cpu)
    if key not in seen:
      seen.add(key)
      cores.append(cpu)
  return cores


def import_reference():
  """Import the reference's own modules from baseline/_ref (never from /root/reference: that path does not exist on
  the GPU box).  `ml_collections` is not installed: its ConfigDict is only used as an attribute dict by the
  reference's config files, so a 6-line stand-in is injected into sys.modules.  Returns the module namespace."""
  import types
  if not os.path.isdir(REF_DIR):
    raise FileNotFoundError(f'{REF_DIR} missing: run tools/install_ref.sh where /root/reference exists')
  if 'ml_collections' not in sys.modules:
    class ConfigDict(dict):
      def __getattr__(self, k):
        try:
          return self[k]
        except KeyError:
          raise AttributeError(k)
      __setattr__ = dict.__setitem__
    m = types.ModuleType('ml_collections')
    m.ConfigDict = ConfigDict
    sys.modules['ml_collections'] = m
  if 'TORCH_EXTENSIONS_DIR' not in os.environ:
    # the two JIT extensions of op/ were pre-built in REF_EXT_DIR; torch takes a lock file in its extension directory
    # even to load them, so they load from a temporary copy and the tree stays untouched (it may be read-only)
    import atexit
    import shutil
    import tempfile
    ext_dir = tempfile.mkdtemp(prefix='score_sde_ref_ext_')
    atexit.register(shutil.rmtree, ext_dir, True)
    if os.path.isdir(REF_EXT_DIR):
      shutil.copytree(REF_EXT_DIR, ext_dir, dirs_exist_ok=True, ignore=shutil.ignore_patterns('lock'))
    os.environ['TORCH_EXTENSIONS_DIR'] = ext_dir
  os.environ.setdefault('TORCH_CUDA_ARCH_LIST', '10.0')
  # our own package has modules of the same names (sampling, sde_lib, ...) under score_sde_pytorch_b200/, never
  # top-level, so putting the reference first on sys.path shadows nothing of ours
  if REF_DIR not in sys.path:
    sys.path.insert(0, REF_DIR)
  import importlib
  ns = types.SimpleNamespace()
  ns.sde_lib = importlib.import_module('sde_lib')
  ns.sampling = importlib.import_module('sampling')
  ns.mutils = importlib.import_module('models.utils')
  ns.ncsnpp = importlib.import_module('models.ncsnpp')            # registers 'ncsnpp'; JIT-loads op/ on first import
  ns.config = importlib.import_module('configs.ve.cifar10_ncsnpp_continuous')
  assert os.path.realpath(ns.sampling.__file__).startswith(os.path.realpath(REF_DIR)), ns.sampling.__file__
  return ns


def reference_pc_steps(batch, steps, warmup):
  """Time PC iterations of the reference itself: its NCSNpp module, its VESDE, and its
  shared_corrector_update_fn / shared_predictor_update_fn called exactly as pc_sampler does (sampling.py:390-409)."""
  ref = import_reference()
  cfg = ref.config.get_config()
  cfg.device = torch.device('cpu')
  cfg.model.init_scale = 1.0
  torch.manual_seed(0)
  model = ref.mutils.get_model(cfg.model.name)(cfg).eval()       # no DataParallel on the CPU
  sde = ref.sde_lib.VESDE(cfg.model.sigma_min, cfg.model.sigma_max, cfg.model.num_scales)
  shape = (batch, 3, 32, 32)
  torch.manual_seed(1)
  x = sde.prior_sampling(shape)
  ts = torch.linspace(sde.T, 1e-5, sde.N)
  pred = ref.sampling.get_predictor(cfg.sampling.predictor.lower())
  corr = ref.sampling.get_corrector(cfg.sampling.corrector.lower())
  times = []
  with torch.no_grad():
    for i in range(warmup + steps):
      t0 = time.perf_counter()
      vec_t = torch.ones(batch) * ts[i]
      x, _ = ref.sampling.shared_corrector_update_fn(x, vec_t, sde, model, corr, True, cfg.sampling.snr, cfg.sampling.n_steps_each)
      x, x_mean = ref.sampling.shared_predictor_update_fn(x, vec_t, sde, model, pred, False, True)
      if i >= warmup:
        times.append(time.perf_counter() - t0)
  assert torch.isfinite(x_mean).all()
  return times, 'reference', dict(x=x, x_mean=x_mean)


def port_pc_steps(batch, steps, warmup):
  """Fallback when baseline/_ref is absent: the oracle port (plain PyTorch fp32 restatement of the same path)."""
  from oracle import ncsnpp_oracle as NO
  from oracle import sampling_oracle as SO
  from score_sde_pytorch_b200.models.ncsnpp import NCSNpp
  cfg = headline_config()
  torch.manual_seed(0)
  sd = NCSNpp(cfg).state_dict()
  model = lambda x, l: NO.ncsnpp_forward(sd, cfg, x, l)
  sde = SO.VE(cfg.model.sigma_min, cfg.model.sigma_max, cfg.model.num_scales)
  shape = (batch, 3, 32, 32)
  torch.manual_seed(1)
  x = sde.prior_sampling(shape)
  ts = torch.linspace(sde.T, 1e-5, sde.N)
  times = []
  with torch.no_grad():
    for i in range(warmup + steps):
      t0 = time.perf_counter()
      vec_t = torch.ones(batch) * ts[i]
      x, _ = SO.langevin_step(sde, model, x, vec_t, cfg.sampling.snr, 1)
      x, x_mean = SO.reverse_diffusion_step(sde, model, x, vec_t)
      if i >= warmup:
        times.append(time.perf_counter() - t0)
  return times, 'port', dict(x=x, x_mean=x_mean)


def cpu_pc_steps(batch, steps, warmup):
  """One CPU-arm measurement in THIS process (threads already pinned by run_reference_arm's re-exec)."""
  threads = int(os.environ.get('B200_BENCH_CPU_THREADS', '0')) or len(physical_cores())
  torch.set_num_threads(threads)
  try:
    times, kind, outputs = reference_pc_steps(batch, steps, warmup)
  except (FileNotFoundError, ImportError) as err:
    print(f'bench: reference unavailable ({err}); timing the oracle port instead', file=sys.stderr)
    times, kind, outputs = port_pc_steps(batch, steps, warmup)
  t_med, t_mean = float(np.median(times)), float(np.mean(times))
  spread = (max(times) - min(times)) / t_med if len(times) > 1 else 0.0
  what = ("the reference's own NCSNpp + shared_corrector_update_fn/shared_predictor_update_fn (baseline/_ref, unmodified)"
          if kind == 'reference' else 'the oracle port (baseline/_ref absent)')
  return dict(value=batch / (N_SAMPLER_STEPS * t_med), unit='images/s', cores=threads, kind=kind,
              sample=f'{steps} PC iterations (2 network evals each) of {what} at batch {batch} after {warmup} warm-up; '
                     f'median {t_med:.3f} s/iteration (mean {t_mean:.3f}, spread {spread:.1%}), extrapolated to '
                     f'{N_SAMPLER_STEPS} iterations; {threads} threads pinned to physical cores',
              host_cpus=os.cpu_count(), ms_per_step=t_med * 1e3, iter_seconds=[round(t, 4) for t in times]), outputs


def pinned_env():
  """Environment for the CPU arm: one OpenMP thread per physical core, bound to it.  torchrun exports
  OMP_NUM_THREADS=1 to every rank (which would reduce the arm to one core), so this overrides it."""
  cores = physical_cores()
  n = min(len(cores), 64)
  env = dict(os.environ)
  env.update(OMP_NUM_THREADS=str(n), MKL_NUM_THREADS=str(n), OMP_PROC_BIND='close', OMP_PLACES='cores',
             GOMP_CPU_AFFINITY=' '.join(str(c) for c in cores[:n]), KMP_AFFINITY='granularity=core,compact',
             B200_BENCH_CPU_THREADS=str(n), B200_BENCH_CPU_PINNED='1', CUDA_VISIBLE_DEVICES='')
  return env


def cpu_arm_subprocess(batch, steps, warmup):
  """Run the CPU arm in a fresh, pinned process (thread pools of the GPU arm's process are already initialised) and
  return its parsed JSON line."""
  cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', str(steps), '--warmup', str(warmup),
         '--cpu-batch', str(batch)]
  env = pinned_env()
  for k in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE', 'MASTER_ADDR', 'MASTER_PORT', 'TORCHELASTIC_RUN_ID'):
    env.pop(k, None)
  out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
  for line in reversed(out.stdout.strip().splitlines()):
    if line.startswith('{'):
      return json.loads(line)
  raise RuntimeError(f'CPU arm produced no JSON line:\n{out.stderr[-2000:]}')


def run_reference_arm(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  if os.environ.get('B200_BENCH_CPU_PINNED') != '1':
    # thread count and binding must be in the environment before libgomp starts: re-exec once
    os.execve(sys.executable, [sys.executable] + sys.argv, pinned_env())
  batch, steps = args.cpu_batch, args.steps
  r, outputs = cpu_pc_steps(batch, steps, max(args.warmup, 1))
  line = dict(impl='reference', metric='PC-sampler images/sec, NCSN++ CIFAR-10 1000-step VE', value=r['value'],
              unit='images/s', n_gpus=args.gpus, steps=steps, warmup=max(args.warmup, 1), ms_per_step=r['ms_per_step'],
              higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic',
              config=dict(workload='NCSN++ cont. CIFAR-10 32x32 VE-SDE PC sampler (1000 steps); CPU arm: bounded sample at '
                                   f'batch {batch}', batch_per_gpu=batch, sampler_steps=N_SAMPLER_STEPS),
              cpu_baseline=dict(value=r['value'], unit='images/s', cores=r['cores'], kind=r['kind'], sample=r['sample'],
                                iter_seconds=r['iter_seconds']),
              e2e=dict(value=r['value'], unit='images/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
              gpu_launches=0)
  print(json.dumps(line), flush=True)
  if args.dump_outputs:
    dump_outputs(args.dump_outputs, outputs)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def load_traffic(precision):
  """DRAM bytes per launch of the contraction kernels from the committed ncu metrics pass of one PC step
  (profiles/traffic_<precision>.json, written by tools/summarize_traffic.py); None when no capture is committed."""
  path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', f'traffic_{precision}.json')
  try:
    k = json.load(open(path))['kernels']
    for name, d in k.items():
      if name.startswith('tcgen05'):
        return round(d['dram_bytes_per_launch'])
  except (OSError, KeyError, ValueError):
    pass
  return None


def measure_tf32_peak(dev, f16=False):
  """cuBLAS GEMM throughput on this device in the operand format the engine computes in: TF32 (kind::tf32
  work) or fp16 with fp32 accumulation (kind::f16 work) - the measured denominator of the tensor roofline."""
  n = 8192
  a = torch.randn(n, n, device=dev)
  b = torch.randn(n, n, device=dev)
  if f16:
    a, b = a.half(), b.half()
  old = torch.backends.cuda.matmul.allow_tf32
  torch.backends.cuda.matmul.allow_tf32 = True
  try:
    for _ in range(3):
      a @ b
    best = 0.0
    for _ in range(6):
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record(); a @ b; e1.record(); torch.cuda.synchronize()
      best = max(best, 2 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
  finally:
    torch.backends.cuda.matmul.allow_tf32 = old
  del a, b
  return best


def check_parity(plan, model, cfg, sde, shape, dev, K, precision):
  from oracle import ncsnpp_oracle as NO, sampling_oracle as SO
  old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
  torch.backends.cudnn.allow_tf32 = False
  torch.backends.cuda.matmul.allow_tf32 = False
  try:
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    osde = SO.VE(cfg.model.sigma_min, cfg.model.sigma_max, cfg.model.num_scales)
    torch.manual_seed(1234)
    x0 = osde.prior_sampling(shape).to(dev)
    B = shape[0]
    # the oracle's eager activations at batch 1024 need several GB per layer: evaluate the network in chunks (the
    # Langevin step size couples the images through batch means of norms, so the LOOP still runs on the full batch)
    chunk = 128

    def net(a, l):
      return torch.cat([NO.ncsnpp_forward(sd, cfg, a[i:i + chunk], l[i:i + chunk]) for i in range(0, B, chunk)])
    torch.cuda.manual_seed(4321)
    t0 = time.perf_counter()
    with torch.no_grad():
      ref, _ = SO.pc_sample(osde, net, shape, eps=1e-5, device=dev, x_init=x0, num_iters=K)
    torch.cuda.synchronize()
    t_oracle = time.perf_counter() - t0
    torch.cuda.manual_seed(4321)
    _, xm = plan.run(x0, first_step=0, num_steps=K)
    a, b = xm.double().flatten(1), ref.double().flatten(1)
    rel = ((a - b).norm(dim=1) / b.norm(dim=1)).cpu().numpy()
    return dict(max_rel_l2=float(rel.max()), p99_rel_l2=float(np.percentile(rel, 99)), median_rel_l2=float(np.median(rel)),
                precision=precision, K=K, batch=B, bound=1e-3,
                oracle='strict-fp32 PyTorch restatement on the same GPU (cudnn/matmul TF32 off), same prior draw and CUDA noise stream',
                oracle_seconds=round(t_oracle, 1))
  finally:
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def timed_steps(plan, x0, warmup, steps):
  plan.run(x0, first_step=0, num_steps=warmup, clone=False)
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  plan.run(x0, first_step=warmup, num_steps=steps, clone=False)
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / steps


def profile_kinds(model, B, dev, x0):
  """Per-kind device time of one eager forward (CUDA events around every launch)."""
  import ctypes
  from score_sde_pytorch_b200 import _lib
  eng = model.engine(B, dev)
  ms_k = (ctypes.c_float * 8)(); fl_k = (ctypes.c_double * 8)(); n_k = (ctypes.c_longlong * 8)()
  xin = x0.clone(); lab = torch.full((B,), 1.0, device=dev); out = torch.empty_like(xin)
  for _ in range(2):
    _lib.call('b200_ncsnpp_profile_forward', eng['h'], _lib.ptr(xin), _lib.ptr(lab), 1, _lib.ptr(out),
              _lib.stream_ptr(dev), ms_k, fl_k, n_k)
  return eng, ms_k, fl_k, n_k


def underfilled_launches(model, B, dev, x0, sms=148):
  """Strong-scaling diagnosis: per-op time at this batch and which contraction launches have fewer tiles than SMs."""
  import ctypes
  from score_sde_pytorch_b200 import _lib
  eng = model.engine(B, dev)
  n = int(_lib.load().b200_ncsnpp_num_ops(eng['h']))
  ms = (ctypes.c_float * n)()
  xin = x0.clone(); lab = torch.full((B,), 1.0, device=dev); out = torch.empty_like(xin)
  for _ in range(2):
    _lib.call('b200_ncsnpp_profile_ops', eng['h'], _lib.ptr(xin), _lib.ptr(lab), 1, _lib.ptr(out), _lib.stream_ptr(dev), ms, n)
  rows = {}
  name = ctypes.create_string_buffer(200); kind = ctypes.c_int(); fl = ctypes.c_double()
  for i in range(n):
    _lib.call('b200_ncsnpp_op_info', eng['h'], i, name, 200, ctypes.byref(kind), ctypes.byref(fl))
    r = rows.setdefault(name.value.decode(), dict(kind=kind.value, launches=0, ms=0.0, flops=0.0))
    r['launches'] += 1; r['ms'] += ms[i]; r['flops'] += fl.value
  out_rows = []
  for k, r in sorted(rows.items(), key=lambda kv: -kv[1]['ms']):
    if r['kind'] != 0:
      continue
    # tiles of a launch: M = B*H*W pixels over 128- (single), 256- (pair / swap) pixel tiles
    import re
    m = re.search(r'@(\d+)', k)
    if not m:
      continue
    res = int(m.group(1))
    px_per_tile = 128 if 'single' in k else 256
    ctas = B * res * res // px_per_tile * (2 if 'pair' in k else 1)
    if 'single128' in k:
      ctas *= 2
    out_rows.append(dict(op=k, launches=r['launches'], ms=round(r['ms'], 4), ctas=ctas, fills_sms=bool(ctas >= sms),
                         tflops=round(r['flops'] / max(r['ms'], 1e-9) / 1e9, 1)))
  return out_rows


def run_gpu_arm(args):
  import torch.distributed as dist
  from score_sde_pytorch_b200 import native, sampling, sde_lib, _lib
  from score_sde_pytorch_b200.models.ncsnpp import NCSNpp
  import ctypes

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  if args.gpus != world and world > 1:
    raise SystemExit(f'--gpus {args.gpus} but WORLD_SIZE={world}')
  dev = torch.device('cuda', local)
  torch.cuda.set_device(dev)
  if world > 1:
    dist.init_process_group('nccl', device_id=dev)

  cfg = headline_config()
  cfg.device = dev
  # weak (headline): args.batch images on every GPU; strong: args.batch images in total, an equal share per GPU
  B = args.batch if args.scaling == 'weak' else max(1, args.batch // world)
  shape = (B, 3, 32, 32)
  torch.manual_seed(0)                       # same random-init weights on every rank ...
  model = NCSNpp(cfg, precision=args.precision, separate_groupnorm=args.separate_groupnorm).to(dev)
  if world > 1:                              # ... and broadcast once over NCCL/NVLink anyway (the production path)
    from score_sde_pytorch_b200 import distributed as bdist
    bdist.broadcast_parameters(model, src=0)
  sde = sde_lib.VESDE(cfg.model.sigma_min, cfg.model.sigma_max, cfg.model.num_scales)
  plan = native.match_pc_plan(sde=sde, model=model, predictor=sampling.ReverseDiffusionPredictor,
                              corrector=sampling.LangevinCorrector, shape=shape, snr=cfg.sampling.snr, n_steps=1,
                              probability_flow=False, continuous=True, eps=1e-5, device=dev)
  assert plan is not None
  torch.manual_seed(1 + rank)                # independent chains per rank
  torch.cuda.manual_seed(1 + rank)
  x_host = sde.prior_sampling(shape).pin_memory()
  out_host = torch.empty(shape).pin_memory()

  # ---- parity at the measured configuration (SURVEY 8d): K PC iterations at the full batch through the engine's
  # plan and through the strict-fp32 GPU oracle, same prior draw, same CUDA noise stream.  The oracle is the checker
  # here, never the thing timed.  Runs on rank 0 only, before any timing; the run FAILS above the north-star bound.
  parity = None
  if rank == 0 and args.parity_steps > 0:
    parity = check_parity(plan, model, cfg, sde, shape, dev, args.parity_steps, args.precision)
    if not (parity['max_rel_l2'] <= 1e-3):
      print(json.dumps(dict(error='parity check failed', parity=parity)), flush=True)
      raise SystemExit(3)

  def barrier():
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  # ---- device-resident timing: K graph replays ----
  x0 = x_host.to(dev)
  plan.run(x0, first_step=0, num_steps=args.warmup, clone=False)  # warm-up (captures the graph)
  clocks = ClockSampler(local)
  barrier()
  clocks.start()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  x, x_mean = plan.run(x0, first_step=args.warmup, num_steps=args.steps, clone=False)
  e1.record()
  barrier()
  clk = clocks.stop()
  ms = e0.elapsed_time(e1)
  finite = bool(torch.isfinite(x_mean).all().item())
  outputs = dict(x=x.cpu(), x_mean=x_mean.cpu()) if args.dump_outputs and rank == 0 else None   # the e2e leg reuses these buffers

  # ---- end to end through the public plan API with host buffers, copies inside the timed region ----
  e2e_steps = args.steps
  barrier()
  f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  f0.record()
  for i in range(e2e_steps):
    # public plan API on host buffers: H2D of the step's input state (pinned), one PC iteration, D2H of the result
    xd, xm = plan.run(x_host, first_step=args.warmup + i, num_steps=1, clone=False)
    out_host.copy_(xm, non_blocking=True)
  f1.record()
  barrier()
  ms_e2e = f0.elapsed_time(f1)

  t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms, ms_e2e = t.tolist()
  ms_per_step = ms / args.steps
  value = world * B / (N_SAMPLER_STEPS * ms_per_step * 1e-3)
  e2e_value = world * B / (N_SAMPLER_STEPS * (ms_e2e / e2e_steps) * 1e-3)

  if rank == 0:
    peaks = load_peaks()
    # ---- per-kind device time of one eager forward (events around every launch) ----
    eng, ms_k, fl_k, n_k = profile_kinds(model, B, dev, x0)
    # algorithmic HBM bytes of the contraction launches (operands once + outputs once), from the plan
    n_ops = int(_lib.load().b200_ncsnpp_num_ops(eng['h']))
    tc_alg_bytes = 0.0
    kind_c, bytes_c = ctypes.c_int(), ctypes.c_double()
    for i in range(n_ops):
      _lib.call('b200_ncsnpp_op_info', eng['h'], i, None, 0, ctypes.byref(kind_c), None)
      if kind_c.value == 0:
        _lib.call('b200_ncsnpp_op_bytes', eng['h'], i, ctypes.byref(bytes_c))
        tc_alg_bytes += bytes_c.value
    kinds = ['tcgen05_contraction', 'cuda_core_contraction', 'groupnorm', 'fir', 'softmax', 'time_embedding', 'misc', 'mma_sync_contraction']
    by_kind = {k: dict(ms=round(ms_k[i], 4), gflop=round(fl_k[i] / 1e9, 2), launches=int(n_k[i])) for i, k in enumerate(kinds)}
    fwd_ms = sum(ms_k[i] for i in range(8))
    tc_ms, tc_flops, tc_n = ms_k[0], fl_k[0], max(int(n_k[0]), 1)
    f16 = args.precision == 'f16'
    tf32_peak = measure_tf32_peak(dev, f16)
    achieved = (tc_flops / tc_n) / ((tc_ms / tc_n) * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    t_hbm_ms = ALG_BYTES_PER_IMG_STEP * B / (peaks['hbm_gbs'] * 1e9) * 1e3
    # Denominators.  fp16 operands run at the bf16 tensor rate, so MEASURED_PEAKS.json's bf16 figures apply directly:
    # per-launch event timing isolates each kernel -> the BURST peak is the fair denominator for `frac`; the whole
    # step is a long back-to-back run -> the SUSTAINED peak for step_tensor_fraction.  TF32 runs at half those rates.
    rate = 1.0 if f16 else 0.5
    burst, sustained = peaks['bf16_tflops'] * rate, peaks['bf16_tflops_sustained'] * rate
    roofline = dict(bound='tensor', kernel=f"gemm_tc_kernel / gemm_tc2_kernel (tcgen05 kind::{'f16' if f16 else 'tf32'} implicit GEMM)",
                    achieved=round(achieved, 2), peak=round(burst, 2), unit='TFLOP/s',
                    frac=round(achieved / burst, 4),
                    peak_source=(f"{peaks['source']}: bf16 burst {peaks['bf16_tflops']} TF/s" + ('' if f16 else ' x 0.5 (TF32 rate)')),
                    frac_of_sustained=round(achieved / sustained, 4), peak_sustained=round(sustained, 2),
                    cublas_in_run=round(tf32_peak, 2), frac_of_cublas_in_run=round(achieved / tf32_peak, 4) if tf32_peak else None,
                    alg_flop_per_launch=tc_flops / tc_n, avg_launch_ms=tc_ms / tc_n, launches_per_forward=tc_n,
                    kernel_share_of_forward=round(tc_ms / fwd_ms, 4) if fwd_ms else None,
                    traffic=load_traffic(args.precision), alg_hbm_bytes_per_launch=round(tc_alg_bytes / tc_n),
                    hbm_fraction_of_step=round(t_hbm_ms / ms_per_step, 4),
                    step_tensor_fraction=round((ALG_FLOP_PER_IMG_STEP * B / (sustained * 1e12) * 1e3) / ms_per_step, 4),
                    step_tflops=round(ALG_FLOP_PER_IMG_STEP * B / (ms_per_step * 1e-3) / 1e12, 1),
                    forward_ms_by_kind=by_kind)
    # ---- the other tensor-core operand format, same model / batch / steps, device-resident timing only ----
    variants = None
    if world == 1 and not args.no_variants and args.precision in ('f16', 'tf32'):
      other = 'tf32' if args.precision == 'f16' else 'f16'
      torch.manual_seed(0)
      model2 = NCSNpp(cfg, precision=other).to(dev)
      plan2 = native.match_pc_plan(sde=sde, model=model2, predictor=sampling.ReverseDiffusionPredictor,
                                   corrector=sampling.LangevinCorrector, shape=shape, snr=cfg.sampling.snr, n_steps=1,
                                   probability_flow=False, continuous=True, eps=1e-5, device=dev)
      ms2 = timed_steps(plan2, x_host.to(dev), args.warmup, args.steps)
      variants = {other: dict(value=round(B / (N_SAMPLER_STEPS * ms2 * 1e-3), 4), unit='images/s', ms_per_step=round(ms2, 4))}
      del plan2, model2
      if args.precision == 'f16':
        # A/B of the two GroupNorm plans in the same run, on the same box (the separate streaming pass of round 1 vs
        # GroupNorm applied on load by the consuming convolution): whichever is not the headline plan is timed here
        torch.manual_seed(0)
        model3 = NCSNpp(cfg, precision='f16', separate_groupnorm=not args.separate_groupnorm).to(dev)
        plan3 = native.match_pc_plan(sde=sde, model=model3, predictor=sampling.ReverseDiffusionPredictor,
                                     corrector=sampling.LangevinCorrector, shape=shape, snr=cfg.sampling.snr, n_steps=1,
                                     probability_flow=False, continuous=True, eps=1e-5, device=dev)
        ms3 = timed_steps(plan3, x_host.to(dev), args.warmup, args.steps)
        variants['f16_groupnorm_' + ('on_load' if args.separate_groupnorm else 'separate_pass')] = dict(
            value=round(B / (N_SAMPLER_STEPS * ms3 * 1e-3), 4), unit='images/s', ms_per_step=round(ms3, 4))
        del plan3, model3
        # A/B of programmatic dependent launch (the headline plan uses the package default)
        torch.manual_seed(0)
        model4 = NCSNpp(cfg, precision='f16', separate_groupnorm=args.separate_groupnorm, pdl=not model.pdl).to(dev)
        plan4 = native.match_pc_plan(sde=sde, model=model4, predictor=sampling.ReverseDiffusionPredictor,
                                     corrector=sampling.LangevinCorrector, shape=shape, snr=cfg.sampling.snr, n_steps=1,
                                     probability_flow=False, continuous=True, eps=1e-5, device=dev)
        ms4 = timed_steps(plan4, x_host.to(dev), args.warmup, args.steps)
        variants['f16_pdl_' + ('off' if model.pdl else 'on')] = dict(value=round(B / (N_SAMPLER_STEPS * ms4 * 1e-3), 4), unit='images/s',
                                                                   ms_per_step=round(ms4, 4))
        del plan4, model4
        # A/B of the halo form of the 3x3 mainloop (headline: package default = swapped AND CTA-pair kernels) against one shifted
        # tile load per filter tap (swapped kernel: in the halo form's chunk-major K order, bit-identical results - round 1's
        # tap-major loop was ~5 % faster than this on those launches, profiles/r02_h1_*; pair kernel: round 1's tap-major
        # loop), and against the halo form in the swapped kernel only
        for hv, key in ((False, 'f16_halo_off_same_k_order'), (True, 'f16_halo_swapped_kernel_only')):
          torch.manual_seed(0)
          model5 = NCSNpp(cfg, precision='f16', separate_groupnorm=args.separate_groupnorm, halo=hv).to(dev)
          plan5 = native.match_pc_plan(sde=sde, model=model5, predictor=sampling.ReverseDiffusionPredictor,
                                       corrector=sampling.LangevinCorrector, shape=shape, snr=cfg.sampling.snr, n_steps=1,
                                       probability_flow=False, continuous=True, eps=1e-5, device=dev)
          ms5 = timed_steps(plan5, x_host.to(dev), args.warmup, args.steps)
          variants[key] = dict(value=round(B / (N_SAMPLER_STEPS * ms5 * 1e-3), 4), unit='images/s', ms_per_step=round(ms5, 4))
          del plan5, model5
    # ---- strong-scaling probe (SURVEY 8e): the same 1024-image job cut over 8 GPUs is 128 images per GPU; time that
    # per-GPU share here and name the launches that under-fill the 148 SMs ----
    strong = None
    if world == 1 and not args.no_strong and B == 1024:
      sb = 128
      splan = native.match_pc_plan(sde=sde, model=model, predictor=sampling.ReverseDiffusionPredictor,
                                   corrector=sampling.LangevinCorrector, shape=(sb, 3, 32, 32), snr=cfg.sampling.snr, n_steps=1,
                                   probability_flow=False, continuous=True, eps=1e-5, device=dev)
      xs = x_host[:sb].to(dev)
      ms_s = timed_steps(splan, xs, args.warmup, args.steps)
      _, msk, _, nk = profile_kinds(model, sb, dev, xs)
      rows = underfilled_launches(model, sb, dev, xs)
      under = [r for r in rows if not r['fills_sms']]
      strong = dict(batch_per_gpu=sb, ms_per_step=round(ms_s, 4), images_per_s_per_gpu=round(sb / (N_SAMPLER_STEPS * ms_s * 1e-3), 4),
                    projected_8gpu_images_per_s=round(8 * sb / (N_SAMPLER_STEPS * ms_s * 1e-3), 4),
                    efficiency_vs_batch_1024=round((sb / ms_s) / (B / ms_per_step), 4),
                    forward_ms_by_kind={k: round(msk[i], 4) for i, k in enumerate(kinds)},
                    underfilled_contractions=dict(count=sum(r['launches'] for r in under), ms=round(sum(r['ms'] for r in under), 4),
                                                  of_total_ms=round(sum(r['ms'] for r in rows), 4), top=under[:8]))
      del splan
    cpu = None
    if world == 1 and not args.no_cpu:
      try:
        cpu = cpu_arm_subprocess(args.cpu_batch, 5, 1)['cpu_baseline']
      except Exception as err:   # the GPU measurement stands on its own; say why the CPU leg is missing
        cpu = dict(value=None, unit='images/s', cores=0, kind='unavailable', sample=f'{type(err).__name__}: {err}'[:300])
    line = dict(metric='PC-sampler images/sec, NCSN++ CIFAR-10 1000-step VE', value=round(value, 4), unit='images/s',
                n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=round(ms_per_step, 4),
                higher_is_better=True, scaling=args.scaling, vs_baseline=None,
                dtype={'tf32': 'tf32', 'f16': 'f16 operands (11-bit significand, as tf32), f32 accumulate and activations', 'fp32': 'f32'}[args.precision],
                data='synthetic',
                config=dict(workload='NCSN++ cont. CIFAR-10 32x32 VE-SDE PC sampler (1000 steps), batch 1024 per GPU'
                            if B == 1024 else f'NCSN++ cont. CIFAR-10 32x32 VE-SDE PC sampler (1000 steps), batch {B} per GPU',
                            batch_per_gpu=B, global_batch=B * world, sampler_steps=N_SAMPLER_STEPS,
                            step='one PC iteration = Langevin corrector + reverse-diffusion predictor (2 score evaluations)',
                            parallelism=f'{world} independent chains shards (weights broadcast once, no in-loop collective)',
                            l2='per-step working set (activations) exceeds the 126 MB L2 by >100x; no explicit flush',
                            weights='random init, init_scale=1, torch.manual_seed(0)', precision=args.precision,
                            groupnorm='separate streaming pass' if args.separate_groupnorm else
                            'applied on load by the consuming convolution where supported (256-channel outputs at 16x16 / 32x32), separate pass elsewhere',
                            conv3x3_mainloop={True: 'halo form (three W-shifted halo copies per channel chunk) in the swapped kernel, one shifted tile per tap in CTA pairs', False: 'one shifted tile load per filter tap', 'pairs': 'halo form in swapped and CTA-pair kernels'}[model.halo]),
                clocks=clk,
                e2e=dict(value=round(e2e_value, 4), unit='images/s', h2d_bytes_per_step=int(np.prod(shape)) * 4,
                         d2h_bytes_per_step=int(np.prod(shape)) * 4, ms_per_step=round(ms_e2e / e2e_steps, 4)),
                gpu_launches=int(plan.launches_per_step()) * args.steps,
                roofline=roofline, finite=finite)
    if variants is not None:
      line['variants'] = variants
    if cpu is not None:
      line['cpu_baseline'] = dict(value=cpu['value'], unit='images/s', cores=cpu['cores'], kind=cpu['kind'], sample=cpu['sample'])
    if strong is not None:
      line['strong_scaling'] = strong
    if parity is not None:
      line['parity'] = parity
    print(json.dumps(line), flush=True)
    if outputs is not None:
      dump_outputs(args.dump_outputs, outputs)
  if world > 1:
    dist.destroy_process_group()


# ---- secondary workloads (SURVEY 8 f2 / f3: the other reference configurations the engine runs) ---------------------------
# `python bench.py --workload NAME` prints ONE JSON line for a non-headline configuration on one GPU: same timing rules
# (device-resident state, CUDA events, >= 3 warm-up steps), no CPU / reference / scaling legs.  Parity for these
# configurations is held by tests/test_gpu_{ddpmpp,progressive,ode}.py; the headline line is unaffected.
def run_secondary_workload(args):
  from score_sde_pytorch_b200 import configs, native, sampling, sde_lib
  from score_sde_pytorch_b200.models.ncsnpp import NCSNpp
  dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', '0')))
  torch.cuda.set_device(dev)
  W = {
    'cifar10_ddpmpp_vp': dict(cfg=configs.vp_cifar10_ddpmpp_continuous, sde=lambda: sde_lib.VPSDE(0.1, 20., 1000), batch=1024, precision='f16',
                              pred=sampling.EulerMaruyamaPredictor, corr=sampling.NoneCorrector, eps=1e-3, snr=0.16, evals=1,
                              desc='DDPM++ cont. CIFAR-10 32x32 VP-SDE, Euler-Maruyama predictor only (configs/vp/cifar10_ddpmpp_continuous.py), 1000 steps'),
    'celebahq_256_ve': dict(cfg=configs.ve_celebahq_256_ncsnpp_continuous, sde=lambda: sde_lib.VESDE(0.01, 348, 2000), batch=16, precision='f16',
                            pred=sampling.ReverseDiffusionPredictor, corr=sampling.LangevinCorrector, eps=1e-5, snr=0.17, evals=2,
                            desc='NCSN++ cont. CelebA-HQ 256x256 VE-SDE PC sampler (configs/ve/celebahq_256_ncsnpp_continuous.py), 2000 steps'),
    'ffhq_1024_ve': dict(cfg=configs.ve_ffhq_1024_ncsnpp_continuous, sde=lambda: sde_lib.VESDE(0.01, 1348, 2000), batch=2, precision='tf32',
                         pred=sampling.ReverseDiffusionPredictor, corr=sampling.LangevinCorrector, eps=1e-5, snr=0.15, evals=2,
                         desc='NCSN++ FFHQ 1024x1024 VE-SDE PC sampler (configs/ve/ffhq_ncsnpp_continuous.py; BASELINE configs[4] per-GPU share), 2000 steps'),
    'celebahq_256_ddpmpp_subvp_ode': dict(cfg=configs.subvp_celebahq_256_ddpmpp_continuous, sde=lambda: sde_lib.subVPSDE(0.1, 20., 1000), batch=8, precision='f16',
                                          ode=True, eps=1e-3,
                                          desc='DDPM++ cont. CelebA-HQ 256 sub-VP probability-flow ODE sampler, RK45 rtol=atol=1e-5, state on the device '
                                               '(BASELINE configs[3] per-GPU share)'),
  }[args.workload]
  cfg = W['cfg']()
  cfg.model.init_scale = 1.0
  cfg.device = dev
  B = W['batch'] if args.batch == 1024 and W['batch'] != 1024 else args.batch
  R = cfg.data.image_size
  shape = (B, 3, R, R)
  torch.manual_seed(0)
  model = NCSNpp(cfg, precision=W['precision']).to(dev)
  sde = W['sde']()
  torch.manual_seed(1); torch.cuda.manual_seed(1)
  clk = ClockSampler(dev.index or 0)
  if W.get('ode'):
    z = sde.prior_sampling(shape).to(dev)
    fn = sampling.get_ode_sampler(sde, shape, lambda v: v, denoise=False, rtol=1e-5, atol=1e-5, eps=W['eps'], device=dev)
    fn(model, z=z.clone())                                     # warm-up solve (plans, allocator)
    torch.cuda.synchronize()
    clk.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    s, nfe = fn(model, z=z.clone())
    e1.record(); torch.cuda.synchronize()
    clocks = clk.stop()
    ms = e0.elapsed_time(e1)
    line = dict(metric='probability-flow ODE sampler images/sec', value=round(B / (ms * 1e-3), 4), unit='images/s', n_gpus=1, steps=int(nfe),
                warmup=1, ms_per_step=round(ms / nfe, 4), higher_is_better=True, scaling='weak', vs_baseline=None, dtype=W['precision'], data='synthetic',
                config=dict(workload=W['desc'], batch_per_gpu=B, nfe=int(nfe), host_scalar_reads=fn.last_stats.get('host_scalar_reads'),
                            step='one right-hand side = one network evaluation + Dormand-Prince stage arithmetic in float64 on the device',
                            weights='random init, init_scale=1, torch.manual_seed(0)'),
                clocks=clocks, finite=bool(torch.isfinite(s).all()), gpu_launches=int(model.launches_per_forward()) * int(nfe))
    outputs = dict(samples=s)
  else:
    plan = native.match_pc_plan(sde=sde, model=model, predictor=W['pred'], corrector=W['corr'], shape=shape, snr=W['snr'], n_steps=1,
                                probability_flow=False, continuous=True, eps=W['eps'], device=dev)
    assert plan is not None
    x0 = sde.prior_sampling(shape).to(dev)
    timed_steps(plan, x0, args.warmup, 1)
    clk.start()
    ms = timed_steps(plan, x0, args.warmup, args.steps)
    clocks = clk.stop()
    N = sde.N
    line = dict(metric='PC-sampler images/sec', value=round(B / (N * ms * 1e-3), 4), unit='images/s', n_gpus=1, steps=args.steps, warmup=args.warmup,
                ms_per_step=round(ms, 4), higher_is_better=True, scaling='weak', vs_baseline=None, dtype=W['precision'], data='synthetic',
                config=dict(workload=W['desc'], batch_per_gpu=B, sampler_steps=N, score_evaluations_per_step=W['evals'],
                            parameters=sum(p.numel() for p in model.parameters()), weights='random init, init_scale=1, torch.manual_seed(0)'),
                clocks=clocks, finite=bool(torch.isfinite(plan._xm).all()), gpu_launches=int(plan.launches_per_step()) * args.steps)
    outputs = dict(x=plan._x, x_mean=plan._xm)     # what plan.run(..., clone=False) handed back in the last timed call
  print(json.dumps(line), flush=True)
  if args.dump_outputs:
    dump_outputs(args.dump_outputs, outputs)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=10)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--batch', type=int, default=1024, help='images per GPU (BASELINE.json configs[1]: 1024)')
  ap.add_argument('--cpu-batch', type=int, default=8, help='batch of the bounded CPU sample')
  ap.add_argument('--precision', default='f16', choices=['tf32', 'f16', 'fp32'],
                  help="tensor-core operand format: 'f16' (default) and 'tf32' both carry 11-bit significands with fp32 "
                       "accumulation and meet the same 1e-3 parity bound (tests/test_gpu_tc.py); 'fp32' = CUDA cores")
  ap.add_argument('--no-variants', action='store_true', help='skip timing the other operand format')
  ap.add_argument('--separate-groupnorm', dest='separate_groupnorm', action='store_true', default=SEPARATE_GROUPNORM_DEFAULT,
                  help='GroupNorm+SiLU as stand-alone streaming passes (round-1 plan)')
  ap.add_argument('--groupnorm-on-load', dest='separate_groupnorm', action='store_false',
                  help='GroupNorm+SiLU applied on load by the consuming convolution where supported (csrc/gemm_tcg.cuh)')
  ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
  ap.add_argument('--no-strong', action='store_true', help='skip the 128-images-per-GPU strong-scaling probe')
  ap.add_argument('--parity-steps', type=int, default=10,
                  help='PC iterations of the in-run parity check against the strict-fp32 GPU oracle at the full batch (0 = skip)')
  ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                  help="'weak' (default, headline): --batch images per GPU; 'strong': --batch images in total, cut over the ranks")
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy')
  ap.add_argument('--workload', default='cifar10_ve',
                  choices=['cifar10_ve', 'cifar10_ddpmpp_vp', 'celebahq_256_ve', 'ffhq_1024_ve', 'celebahq_256_ddpmpp_subvp_ode'],
                  help="'cifar10_ve' (default) is the headline line; the others print one line for a secondary configuration (1 GPU)")
  args = ap.parse_args()
  if args.warmup < 3 and args.impl == 'ours':
    args.warmup = 3
  if args.impl == 'reference':
    run_reference_arm(args)
  elif args.workload != 'cifar10_ve':
    run_secondary_workload(args)
  else:
    run_gpu_arm(args)


if __name__ == '__main__':
  main()
