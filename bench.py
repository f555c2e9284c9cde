"""Benchmark of the render hot path (NerfModel.__call__) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--precision P] [--workload W]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...      # the reference's CPU path (oracle port)
  python bench.py --dump-outputs DIR ...    # also write the last timed step's outputs as .npy

Metric (BASELINE.json): ray-samples/sec, coarse+fine, device-timed; PSNR vs ref.
One ray-sample = one (warp MLP + NeRF MLP) point evaluation; a ray costs
Nc + (Nc + Nf) of them (SURVEY.md §8d).  A step = one forward of the whole
pipeline over one batch of synthetic rays.  Default workload: the north-star
synthetic (65,536 rays x (128+128) samples, gpu_quarterhd.gin model dimensions)
per GPU; rays shard across GPUs with no data-path collective (weak scaling).

The headline (`value`, `e2e`, `roofline`) is measured in the PARITY-HOLDING
tensor-core mode (precision fp16x3: 1e-4 per stage against the reference's fp32
arithmetic); the bf16 mode's throughput and its measured error are reported next
to it under `also`.  After the timed region the line's `parity` object compares a
sample of the rays that were just timed with the oracle (max-rel errors, PSNR); a
run whose errors exceed the mode's stated bound exits non-zero.

One JSON line is printed by rank 0 (see the task contract for the keys).
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
  sys.path.insert(0, REPO)

NEAR, FAR = 0.02, 0.83
N_IDS = 200

# SURVEY.md §8(d) workloads: model dimensions of the gin files, forward FLOP per
# ray-sample = 2 x (warp MLP + NeRF MLP MACs); padding / emulation passes not counted.
WORKLOADS = {
    'northstar': dict(
        rays=65536, nc=128, nf=128, fp=8, fw=8, app=True, cam=False, flop=1370112,
        desc='north-star synthetic: {B} rays/GPU x (128+128) samples = 384 ray-samples/ray, '
             'gpu_quarterhd.gin model dims'),
    'quarterhd-train': dict(
        rays=6144, nc=128, nf=128, fp=8, fw=8, app=True, cam=False, flop=1370112,
        desc='gpu_quarterhd.gin training batch: {B} rays x (128+128) samples'),
    'vrig-train': dict(
        rays=6144, nc=128, nf=128, fp=8, fw=6, app=False, cam=True, flop=1364480,
        desc='gpu_vrig_paper.gin batch: {B} rays x (128+128) samples, num_warp_freqs=6, '
             'camera metadata (rgb condition 29)'),
    'fullhd-train': dict(
        rays=4096, nc=256, nf=256, fp=10, fw=8, app=True, cam=False, flop=1382400,
        desc='gpu_fullhd.gin training batch: {B} rays x (256+256) samples, num_nerf_point_freqs=10'),
    'eval-1080p': dict(
        rays=1920 * 1080, nc=256, nf=256, fp=10, fw=8, app=True, cam=False, flop=1382400,
        frame=(1920, 1080),
        desc='eval.py render path: one full 1920x1080 frame = {B} rays x (256+256) samples, '
             'gpu_fullhd.gin model dims, rays generated on the GPU per rank, frame split over '
             'the ranks, one all_gather of 24 B/ray'),
    'quarterhd-trainstep': dict(
        rays=6144, nc=128, nf=128, fp=8, fw=8, app=True, cam=False, flop=1370112, trainstep=True,
        desc='training.train_step on the gpu_quarterhd.gin batch: {B} rays per GPU x (128+128) samples (global '
             'batch 6144 split over the ranks as the reference does): value_and_grad of the photometric loss '
             '(fp32, layer-wise tape), ONE NCCL all_reduce of the flat gradient, Adam'),
    'vrig-trainstep': dict(
        rays=6144, nc=128, nf=128, fp=8, fw=6, app=False, cam=True, flop=1364480, trainstep=True, reg=True,
        desc='training.train_step as gpu_vrig_paper.gin configures it: {B} rays per GPU x (128+128) samples, '
             "elastic loss on the warp Jacobian of every coarse sample (elastic_reduce_method='weight', log_svals), "
             'background loss on {B} points, photometric loss; ONE NCCL all_reduce of the flat gradient, Adam'),
    'fullhd-65536': dict(
        rays=65536, nc=256, nf=256, fp=10, fw=8, app=True, cam=False, flop=1382400,
        desc='gpu_fullhd.gin model dims at {B} rays x (256+256) samples'),
}

# Stated parity bounds per mode, metric |a-b| / (|b| + 1e-2) (absolute below 1e-2).
#   coarse      : coarse level, well conditioned              (the 1e-4 gate)
#   fine_oracle_z: fine level evaluated on the oracle's z     (the 1e-4 gate)
#   e2e         : fine level end to end; inverse-CDF resampling amplifies fp32
#                 round-off in empty space (DESIGN.md §2), stated 2e-3
PARITY_BOUNDS = {
    'fp32': dict(coarse=1e-4, fine_oracle_z=1e-4, e2e=2e-3, psnr_db=70.0),
    'fp16x3': dict(coarse=1e-4, fine_oracle_z=1e-4, e2e=2e-3, psnr_db=70.0),
    'bf16': dict(coarse=8e-2, fine_oracle_z=8e-2, e2e=1.5e-1, psnr_db=35.0),
}
DTYPE_NAMES = {
    'fp32': 'fp32',
    'bf16': 'bf16',
    'fp16x3': 'fp16x3 (fp32 emulated on tcgen05: 3 fp16 MMA chains, fp32 accumulate)',
}


def parse_args():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=5)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--workload', default='northstar', choices=sorted(WORKLOADS))
  ap.add_argument('--rays', type=int, default=None, help='rays per GPU per step (default: the workload\'s)')
  ap.add_argument('--precision', default=None, choices=[None, 'fp32', 'bf16', 'fp16x3'],
                  help='headline mode (default: fp16x3, the parity-holding tensor-core mode)')
  ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                  help='weak: --rays per GPU; strong: --rays in total, split over the ranks')
  ap.add_argument('--no-also', action='store_true', help='skip the secondary modes / strong-scaling extras')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-parity', action='store_true')
  ap.add_argument('--cpu-seconds', type=float, default=15.0)
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='after the timed steps, write what the last timed step returned (rank 0) '
                       'as DIR/<name>.npy')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'b200':
    ap.error('--dump-outputs writes the outputs of the b200 arm')
  return args


DUMP_MAX_BYTES = 60 * 2**20      # the .npy files of one dump stay under 64 MB together


def dump_outputs(out_dir, arrays):
  """Writes {name: tensor} as out_dir/<name>.npy (float32, or float64 where the tensor is).
  Inputs are seeded, so two builds' dumps of the same command compare element for element.
  Above DUMP_MAX_BYTES in all, every array keeps the same fixed, seeded sample of its
  leading dimension (arrays with the same leading size keep the same rows)."""
  import numpy as np
  import torch
  arrays = {k: v.detach().cpu().to(torch.float64 if v.dtype == torch.float64 else torch.float32)
            for k, v in arrays.items()}
  total = sum(v.numel() * v.element_size() for v in arrays.values())
  if total > DUMP_MAX_BYTES:
    keep = DUMP_MAX_BYTES / total
    for k, v in arrays.items():
      if v.dim() == 0:
        continue
      n = v.shape[0]
      idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:max(1, int(n * keep))]
      arrays[k] = v[idx.sort().values]
  os.makedirs(out_dir, exist_ok=True)
  for k, v in arrays.items():
    np.save(os.path.join(out_dir, k + '.npy'), v.numpy())


def flat_outputs(tree, prefix=''):
  """{'coarse': {'rgb': t, ...}, ...} -> {'coarse_rgb': t, ...} (tensor and number leaves; '/' -> '_')."""
  import torch
  flat = {}
  for k, v in tree.items():
    name = prefix + k.replace('/', '_')
    if isinstance(v, dict):
      flat.update(flat_outputs(v, name + '_'))
    elif torch.is_tensor(v):
      flat[name] = v
    elif isinstance(v, (int, float)):
      flat[name] = torch.tensor(float(v), dtype=torch.float64)
  return flat


def oracle_spec(wl):
  from oracle import nerfies_oracle as O
  return O.OracleSpec(
      num_coarse_samples=wl['nc'], num_fine_samples=wl['nf'], near=NEAR, far=FAR,
      num_nerf_point_freqs=wl['fp'], num_warp_freqs=wl['fw'], sigma_activation='softplus',
      use_warp=True, warp_field_type='se3', use_appearance_metadata=wl['app'],
      use_camera_metadata=wl['cam'], num_warp_embeddings=N_IDS,
      num_appearance_embeddings=N_IDS if wl['app'] else 1,
      num_camera_embeddings=2 if wl['cam'] else 1)


def model_config(wl):
  import nerfies_b200 as nb
  # gpu_*.gin (+ warp_defaults.gin, defaults.gin) model fields; the deterministic
  # path (eval.py:239).
  return nb.configs.ModelConfig(
      use_stratified_sampling=False, use_viewdirs=True, use_warp=True,
      warp_field_type='se3', num_warp_freqs=wl['fw'], num_warp_features=8,
      use_appearance_metadata=wl['app'], use_camera_metadata=wl['cam'],
      camera_metadata_dims=2, sigma_activation='softplus',
      num_nerf_point_freqs=wl['fp'], nerf_trunk_width=256, nerf_trunk_depth=8,
      num_coarse_samples=wl['nc'], num_fine_samples=wl['nf'])


def trained_like(params, scale=3.0, bias_std=0.1, seed=1):
  """"Trained-like" random weights (SURVEY §8d): hidden kernels x1.3, heads xscale,
  the density head x4*scale, small non-zero warp heads, N(0, bias_std) biases - so
  that sigma / alpha / the resampled PDF are non-degenerate.  The same recipe (and
  the same torch CPU generator stream) as the oracle's test helper, restated here so
  that the product arm does not import oracle/ for its inputs."""
  import torch
  gen = torch.Generator().manual_seed(seed)

  def rec(t, path):
    if isinstance(t, dict):
      return {k: rec(v, path + (k,)) for k, v in t.items()}
    if 'warp_field' in path and path[-2] == 'logit':
      if path[-1] == 'kernel':
        return (torch.rand(t.shape, generator=gen) * 2 - 1) * 2e-3
      return (torch.rand(t.shape, generator=gen) * 2 - 1) * 1e-2
    if path[-1] == 'kernel':
      if path[-2] == 'logit' and 'MLP_2' in path:
        return t * (4.0 * scale)
      if path[-2] == 'logit':
        return t * scale
      return t * 1.3
    if path[-1] == 'bias':
      return torch.randn(t.shape, generator=gen) * bias_std
    return t

  return rec(params, ())


def synthetic_rays(num_rays, seed, wl):
  """SURVEY.md §8(d) synthetic inputs, float32, seeded."""
  import torch
  g = torch.Generator().manual_seed(seed)
  origins = torch.rand(num_rays, 3, generator=g) - 0.5
  d = torch.randn(num_rays, 3, generator=g)
  directions = d / torch.linalg.norm(d, dim=-1, keepdim=True)
  md = {'warp': torch.randint(0, N_IDS, (num_rays, 1), generator=g, dtype=torch.int32),
        'appearance': torch.randint(0, N_IDS, (num_rays, 1), generator=g, dtype=torch.int32),
        'camera': torch.randint(0, 2, (num_rays, 1), generator=g, dtype=torch.int32)}
  if not wl['app']:
    md.pop('appearance')
  if not wl['cam']:
    md.pop('camera')
  return {'origins': origins, 'directions': directions, 'metadata': md}


class ClockSampler:
  """nvidia-smi clocks / throttle reasons during the timed region."""
  FIELDS = ('clocks.sm,clocks.max.sm,power.draw,'
            'clocks_event_reasons.hw_slowdown,'
            'clocks_event_reasons.hw_thermal_slowdown,'
            'clocks_event_reasons.sw_thermal_slowdown,'
            'clocks_event_reasons.sw_power_cap')

  def __init__(self, index):
    self.index, self.rows, self.proc = index, [], None

  def start(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.FIELDS}',
           '--format=csv,noheader,nounits', '-lms', '100'],
          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except OSError:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([c.strip() for c in line.split(',')])

  def stop(self):
    if not self.proc:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except subprocess.TimeoutExpired:
      self.proc.kill()
    sm, mx, reasons, pw = [], None, set(), []
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
             'sw_power_cap']
    for r in self.rows:
      if len(r) < 7:
        continue
      try:
        sm.append(float(r[0]))
        mx = float(r[1])
      except ValueError:
        continue
      try:
        pw.append(float(r[2]))
      except ValueError:
        pass
      for n, v in zip(names, r[3:7]):
        if v.lower().startswith('active'):
          reasons.add(n)
    busy = [v for v in sm if mx and v > 0.3 * mx] or sm
    return {'sm_mhz': statistics.median(busy) if busy else None,
            'sm_max_mhz': mx, 'reasons': sorted(reasons),
            'samples': len(sm), 'power_w': max(pw) if pw else None,
            'power_w_median': statistics.median(pw) if pw else None}


# ----------------------------------------------------------------------------
# CPU legs: the reference's algorithm on the host (oracle port).
# ----------------------------------------------------------------------------
def time_oracle(num_rays, threads, wl, seed=0):
  """Seconds for one oracle forward of `num_rays` rays (torch CPU fp32)."""
  import torch
  from oracle import nerfies_oracle as O
  spec = oracle_spec(wl)
  torch.set_num_threads(threads)
  params = O.make_trained_like(O.init_params(spec, seed), seed=seed + 1)
  rays = O.synthetic_rays(num_rays, spec, seed=seed + 2)
  chunk = 256   # bounds the (B, Nc-1, Nf) mask of sample_pdf and activations
  t0 = time.perf_counter()
  with torch.no_grad():
    for s in range(0, num_rays, chunk):
      sub = {'origins': rays['origins'][s:s + chunk],
             'directions': rays['directions'][s:s + chunk],
             'metadata': {k: v[s:s + chunk] for k, v in rays['metadata'].items()}}
      O.render_forward(params, spec, sub, warp_alpha=float(wl['fw']))
  return time.perf_counter() - t0


def best_thread_count(wl):
  """torch's intra-op pool does not scale to every core on large hosts (128
  threads on the GPU box is ~30x slower than 8-32): probe a few counts on a small
  sample and keep the fastest.  Returns (threads, rays_per_second)."""
  cores = os.cpu_count() or 1
  cands = sorted({c for c in (cores, 64, 32, 16, 8) if c <= cores})
  time_oracle(128, cands[0], wl)                 # warm-up (thread pools, MKL)
  best = None
  for c in cands:
    t = time_oracle(128, c, wl)
    if best is None or t < best[1]:
      best = (c, t)
  return best[0], 128 / best[1]


def _oracle_worker(idx, wl_name, threads, max_rays, seed, barrier, cmd_q, out_q):
  """One host process of the multi-process CPU leg: its own torch thread pool, its
  own shard of the rays.  Commands: n > 0 = render n rays (timed between the barrier
  and the end of the loop), 0 = exit."""
  try:
    import torch
    from oracle import nerfies_oracle as O
    wl = WORKLOADS[wl_name]
    spec = oracle_spec(wl)
    torch.set_num_threads(threads)
    params = O.make_trained_like(O.init_params(spec, seed), seed=seed + 1)
    rays = O.synthetic_rays(max_rays, spec, seed=seed + 2 + idx)
    chunk = 256

    def run(n):
      with torch.no_grad():
        for s in range(0, n, chunk):
          e = min(n, s + chunk)
          sub = {'origins': rays['origins'][s:e], 'directions': rays['directions'][s:e],
                 'metadata': {k: v[s:e] for k, v in rays['metadata'].items()}}
          O.render_forward(params, spec, sub, warp_alpha=float(wl['fw']))
    run(64)                                        # thread pool, MKL, allocator warm-up
    out_q.put((idx, 'ready', 0.0, 0.0))
    while True:
      n = cmd_q.get(timeout=900)
      if n <= 0:
        return
      barrier.wait(timeout=300)
      t0 = time.perf_counter()
      run(min(n, max_rays))
      out_q.put((idx, 'done', t0, time.perf_counter()))
  except Exception as e:                           # the parent falls back to the single-process layout
    try:
      barrier.abort()
    except Exception:
      pass
    out_q.put((idx, 'error: ' + repr(e), 0.0, 0.0))


class OraclePool:
  """cores // threads host processes, each a torch-CPU oracle with `threads` intra-op
  threads on its own shard of the rays: the data-parallel layout the reference itself
  uses across devices, here across the host's cores (one torch process stops scaling at
  16-32 threads).  run(n) = wall seconds for every process to render n rays concurrently
  (CLOCK_MONOTONIC is system-wide: earliest start to latest end)."""

  def __init__(self, procs, threads, wl_name, max_rays, seed=0):
    import multiprocessing as mp
    ctx = mp.get_context('spawn')                  # never fork a process that may hold a CUDA context
    self.procs, self.ok = procs, False
    self.barrier, self.out_q = ctx.Barrier(procs), ctx.Queue()
    self.cmd_qs = [ctx.Queue() for _ in range(procs)]
    self.ps = [ctx.Process(target=_oracle_worker,
                           args=(i, wl_name, threads, max_rays, seed, self.barrier, self.cmd_qs[i], self.out_q),
                           daemon=True) for i in range(procs)]
    for p in self.ps:
      p.start()
    try:
      self.ok = all(self.out_q.get(timeout=600)[1] == 'ready' for _ in self.ps)
    except Exception:
      self.ok = False

  def run(self, n):
    if not self.ok:
      return None
    for q in self.cmd_qs:
      q.put(n)
    try:
      res = [self.out_q.get(timeout=900) for _ in self.ps]
    except Exception:
      self.ok = False
      return None
    if any(r[1] != 'done' for r in res):
      self.ok = False
      return None
    return max(r[3] for r in res) - min(r[2] for r in res)

  def close(self):
    for q in self.cmd_qs:
      try:
        q.put(0)
      except Exception:
        pass
    for p in self.ps:
      p.join(timeout=20)
      if p.is_alive():
        p.terminate()                              # our own child, by handle


class CpuLayout:
  """The faster of (one process x the best thread count) and (cores // threads processes x
  that thread count) for the reference's algorithm on this host; sample(budget) times one
  bounded sample of the workload with it."""

  def __init__(self, wl_name, max_rays):
    self.wl_name, self.wl, self.max_rays = wl_name, WORKLOADS[wl_name], max_rays
    self.threads, self.rate = best_thread_count(self.wl)          # rays/s, one process
    self.pool, self.procs = None, 1
    procs = (os.cpu_count() or 1) // self.threads
    if procs >= 2:
      pool = OraclePool(procs, self.threads, wl_name, max_rays)
      t = pool.run(256)
      if t and procs * 256 / t > self.rate:
        self.pool, self.procs, self.rate = pool, procs, procs * 256 / t
      else:
        pool.close()

  def sample(self, budget_s):
    """-> (ray-samples/s, host threads used, rays, seconds, description)"""
    evals = 2 * self.wl['nc'] + self.wl['nf']
    if self.pool:
      per = int(min(self.max_rays, max(256, self.rate / self.procs * budget_s)) // 256 * 256)
      t = self.pool.run(per)
      if t:
        n = per * self.procs
        return (n * evals / t, self.procs * self.threads, n, t,
                f'{n} rays sharded over {self.procs} processes x {self.threads} torch threads')
      self.pool, self.procs = None, 1                # a worker died: fall back
      self.threads, self.rate = best_thread_count(self.wl)
    n = int(min(self.max_rays, max(256, self.rate * budget_s)) // 256 * 256)
    t = time_oracle(n, self.threads, self.wl)
    return (n * evals / t, self.threads, n, t, f'{n} rays, one process x {self.threads} torch threads')

  def close(self):
    if self.pool:
      self.pool.close()


def cpu_baseline(budget_s, wl_name):
  """The reference's algorithm on the host cores (oracle port; the JAX original
  cannot run in this image), on a bounded sample of the same workload."""
  wl = WORKLOADS[wl_name]
  lay = CpuLayout(wl_name, 4096)
  try:
    value, used, n, t, how = lay.sample(budget_s)
  finally:
    lay.close()
  return {'value': value, 'unit': 'ray-samples/s',
          'cores': used, 'kind': 'port',
          'sample': f'{how} x ({wl["nc"]}+{wl["nf"]}) samples of the workload, '
                    f'torch-CPU fp32 oracle, {t:.1f} s; {used} of '
                    f'{os.cpu_count()} host threads (the faster of one process and ray-sharded processes)'}


def workload_text(wl, B):
  return (wl['desc'].format(B=B) + ', SE(3) warp on, deterministic sampling, '
          'trained-like random weights')


def run_reference(args):
  """--impl reference: the reference's CPU path (oracle port), all host threads,
  each step a bounded sample of the workload."""
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  wl = WORKLOADS[args.workload]
  B = args.rays or wl['rays']
  evals = 2 * wl['nc'] + wl['nf']
  # every step = one bounded sample of the workload on all the host cores; the whole run stays
  # within a few minutes whatever --steps is
  lay = CpuLayout(args.workload, 4096)
  per_step = max(1.0, min(8.0, 150.0 / max(1, args.steps + min(args.warmup, 1))))
  try:
    for _ in range(min(args.warmup, 1)):
      lay.sample(per_step)
    legs = [lay.sample(per_step) for _ in range(args.steps)]
  finally:
    lay.close()
  value = sum(l[0] for l in legs) / len(legs)
  threads, n = legs[-1][1], legs[-1][2]
  sec = sum(l[3] for l in legs) / len(legs)
  line = {
      # same metric / unit / workload as the b200 arm (host-timed: there is no device)
      'impl': 'reference', 'metric': 'ray-samples/sec (coarse+fine, device-timed)',
      'value': value, 'unit': 'ray-samples/s', 'n_gpus': args.gpus,
      'steps': args.steps, 'warmup': min(args.warmup, 1),
      'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': args.scaling,
      'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
      'config': {'workload': workload_text(wl, B) + f'; each step a bounded sample of {n} rays '
                             'of it on the host CPU',
                 'rays_per_step': n, 'precision': 'fp32',
                 'timing': 'host wall clock around the reference algorithm (oracle port)'},
      'cpu_baseline': {'value': value, 'unit': 'ray-samples/s',
                       'cores': threads, 'kind': 'port',
                       'sample': f'{legs[-1][4]} per step; restated reference on '
                                 'torch-CPU fp32 (JAX/Flax not installable)'},
      'e2e': {'value': value, 'unit': 'ray-samples/s', 'h2d_bytes_per_step': 0,
              'd2h_bytes_per_step': 0},
      'gpu_launches': 0,
  }
  emit(line)


# ----------------------------------------------------------------------------
# The b200 arm
# ----------------------------------------------------------------------------
def rel_err(a, b, floor=1e-2):
  a, b = a.double(), b.double()
  return float(((a - b).abs() / (b.abs() + floor)).max())


def psnr_db(a, b):
  """utils.compute_psnr (utils.py:94-103): -10 log10(mse)."""
  mse = float(((a.double() - b.double())**2).mean())
  return -10.0 * math.log10(max(mse, 1e-20))


def parity_check(model, variables, params_cpu, rays_host, out, wl, precision, n_sample=256):
  """Compares a sample of the rays that were just timed with the oracle
  (BASELINE.json: "PSNR vs ref"): the step's own outputs for the coarse level and
  end to end, plus the fine level re-evaluated on the oracle's z (the
  well-conditioned per-stage check)."""
  import torch
  from oracle import nerfies_oracle as O   # the checker, outside every timed region
  from nerfies_b200.models import _prep_f32, _prep_ids, _ptr, _stream
  from nerfies_b200 import _lib
  spec = oracle_spec(wl)
  B = rays_host['origins'].shape[0]
  n = min(n_sample, B)
  idx = torch.linspace(0, B - 1, n).round().long()
  sub = {'origins': rays_host['origins'][idx], 'directions': rays_host['directions'][idx],
         'metadata': {k: v[idx] for k, v in rays_host['metadata'].items()}}
  alpha = float(wl['fw'])
  torch.set_num_threads(min(16, os.cpu_count() or 1))
  with torch.no_grad():
    ref = O.render_forward(params_cpu, spec, sub, warp_alpha=alpha, return_points=True)
  dev = model.device
  got = {lv: {k: out[lv][k][idx.to(dev)].cpu() for k in ('rgb', 'depth', 'acc')}
         for lv in ('coarse', 'fine')}
  res = {'rays': n, 'metric': 'max |a-b| / (|b| + 1e-2) vs the fp32 oracle (oracle/nerfies_oracle.py)'}
  res['coarse'] = {f'max_rel_{k}': rel_err(got['coarse'][k], ref['coarse'][k]) for k in ('rgb', 'depth', 'acc')}
  res['e2e'] = {f'max_rel_{k}': rel_err(got['fine'][k], ref['fine'][k]) for k in ('rgb', 'depth', 'acc')}
  res['e2e']['psnr_db'] = psnr_db(got['fine']['rgb'], ref['fine']['rgb'])
  # fine level on the oracle's z through nfb_render_samples
  hd = model.handle(B)
  z = ref['fine']['z_vals'].contiguous()
  S = z.shape[1]
  o = _prep_f32(sub['origins'], dev)
  d = _prep_f32(sub['directions'], dev)
  ids = [_prep_ids(sub['metadata'].get(k), dev) for k in ('warp', 'appearance', 'camera')]
  zc = _prep_f32(z, dev)
  buf = torch.empty(n, 6, device=dev)
  _lib.check(hd.lib.nfb_render_samples(
      hd.h, 1, n, S, _ptr(zc), _ptr(o), _ptr(d), None, _ptr(ids[0]), _ptr(ids[1]), _ptr(ids[2]),
      alpha, 0, _ptr(buf), None, None, None, _stream()))
  torch.cuda.synchronize()
  buf = buf.cpu()
  fz = {'rgb': buf[:, :3], 'depth': buf[:, 3], 'acc': buf[:, 5]}
  res['fine_oracle_z'] = {f'max_rel_{k}': rel_err(fz[k], ref['fine'][k]) for k in ('rgb', 'depth', 'acc')}
  res['fine_oracle_z']['psnr_db'] = psnr_db(fz['rgb'], ref['fine']['rgb'])
  bounds = PARITY_BOUNDS[precision]
  ok = all(max(v for k, v in res[s].items() if k.startswith('max_rel')) < bounds[s]
           for s in ('coarse', 'fine_oracle_z', 'e2e'))
  ok = ok and res['e2e']['psnr_db'] > bounds['psnr_db']
  res['bounds'] = bounds
  res['ok'] = bool(ok)
  return res


def measure(precision, wl, B, args, ctx, want_parity):
  """Times `args.steps` forwards of B rays per rank in one precision mode."""
  import torch
  import torch.distributed as dist
  import nerfies_b200 as nb
  dev, world, rank, local_rank = ctx['dev'], ctx['world'], ctx['rank'], ctx['local_rank']
  evals = 2 * wl['nc'] + wl['nf']
  model, params = nb.construct_nerf(0, model_config(wl), B, range(N_IDS), range(2),
                                    range(N_IDS), NEAR, FAR,
                                    precision=precision, device=dev)
  cpu = lambda t: ({k: cpu(v) for k, v in t.items()} if isinstance(t, dict)
                   else t.cpu())
  gpu = lambda t: ({k: gpu(v) for k, v in t.items()} if isinstance(t, dict)
                   else t.to(dev))
  params_cpu = trained_like(cpu(params), seed=1)
  params = gpu(params_cpu)
  rays_host = synthetic_rays(B, 1000 + rank, wl)   # each rank its own rays
  rays = {'origins': rays_host['origins'].to(dev),
          'directions': rays_host['directions'].to(dev),
          'metadata': {k: v.to(dev) for k, v in rays_host['metadata'].items()}}
  variables = {'params': params}
  warp_extra = {'alpha': float(wl['fw']), 'time_alpha': 0.0}
  flush = ctx['flush']

  def step():
    return model.apply(variables, rays, warp_extra=warp_extra)

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  for _ in range(max(args.warmup, 3)):
    out = step()
  hd = model.handle(B)
  _ = hd.lib.nfb_set_profiling(hd.h, 1)
  barrier()
  sampler = ClockSampler(local_rank)
  sampler.start()
  launches0 = model.kernel_launches()
  ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        for _ in range(args.steps)]
  field_ms = []
  barrier()
  wall0 = time.perf_counter()
  for i in range(args.steps):
    flush.zero_()                      # L2 flush between timed iterations
    ev[i][0].record()
    out = step()
    ev[i][1].record()
    ev[i][1].synchronize()
    field_ms.append((float(hd.lib.nfb_field_time_ms(hd.h, 0)),
                     float(hd.lib.nfb_field_time_ms(hd.h, 1))))
  barrier()
  wall = time.perf_counter() - wall0
  launches = model.kernel_launches() - launches0
  clocks = sampler.stop()
  hd.lib.nfb_set_profiling(hd.h, 0)
  step_ms = [a.elapsed_time(b) for a, b in ev]
  total_ms = torch.tensor([sum(step_ms)], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
  ms_per_step = float(total_ms) / args.steps
  res = {
      'precision': precision, 'ms_per_step': ms_per_step,
      'value': world * B * evals / (ms_per_step * 1e-3),
      'launches': int(launches), 'clocks': clocks, 'wall': wall,
      'field_ms': (statistics.mean(m[0] for m in field_ms), statistics.mean(m[1] for m in field_ms)),
      'out': out,
  }
  if want_parity and rank == 0:
    res['parity'] = parity_check(model, variables, params_cpu, rays_host, out, wl, precision)
  res['model'], res['variables'], res['rays_host'], res['warp_extra'] = model, variables, rays_host, warp_extra
  return res


def roofline(res, wl, B, peaks, precision):
  fc, ff = res['field_ms']
  fine_flop = B * (wl['nc'] + wl['nf']) * wl['flop']
  achieved = fine_flop / (ff * 1e-3) / 1e12
  # a step is tens of milliseconds between flushes and syncs: the burst cuBLAS peak
  # is the denominator (VERDICT r01); the sustained one is quoted beside it.
  peak = peaks.get('bf16_tflops') or peaks.get('bf16_tflops_sustained')
  peak_src = 'measured (MEASURED_PEAKS.json, burst bf16 cuBLAS 8192^3)'
  if not peak:
    peak, peak_src = 1590.0, 'fallback (B200_PROFILING.md)'
  traffic = None
  try:
    with open(os.path.join(REPO, 'profiles', 'traffic.json')) as f:
      traffic = json.load(f).get(precision, {}).get('field_fine_dram_bytes')
  except (OSError, ValueError):
    pass
  notes = {
      'fp32': 'fp32 mode runs on the FFMA pipe; the fraction is still quoted against the bf16 '
              'tensor peak the north-star names',
      'fp16x3': 'ALGORITHMIC FLOPs only: the three fp16 MMA chains that emulate fp32 execute 3x '
                'this many tensor FLOPs (no credit taken); tensor-pipe busy fraction = 3 x frac. '
                'The kernel runs at the board power limit (see clocks: sw_power_cap, ~1.75 of '
                '1.965 GHz, ~990 W in a 60-step run: profiles/r02_ab_x3_variants.txt), so the '
                'fraction is bounded by energy per MMA, not by the issue rate',
      'bf16': '',
  }
  r = {
      'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
      'frac': achieved / peak, 'traffic': traffic,
      'kernel': f'field kernel, fine level ({B * (wl["nc"] + wl["nf"])} rows x {wl["flop"]} FLOP)',
      'kernel_ms': ff, 'coarse_kernel_ms': fc,
      'share_of_step': (fc + ff) / res['ms_per_step'],
      'peak_source': peak_src, 'note': notes[precision],
  }
  if peaks.get('bf16_tflops_sustained'):
    r['frac_of_sustained_peak'] = achieved / peaks['bf16_tflops_sustained']
  if precision == 'fp16x3':
    r['tensor_pipe_frac_executed'] = 3 * achieved / peak
    if peaks.get('bf16_tflops_sustained'):
      # the power-limited tensor rate of the chip (cuBLAS bf16 back to back for 4 s runs at ~1.34 GHz under
      # the same 1000 W cap) is the bound this kernel actually meets: executed FLOPs / sustained peak
      r['tensor_pipe_frac_executed_of_sustained'] = 3 * achieved / peaks['bf16_tflops_sustained']
  return r


def measure_eval_frame(args, wl, precision, ctx, steps, dump_dir=None):
  """BASELINE.json's fifth config (eval.py:330-353): a full frame, rays split
  1 -> N GPUs, forward only.  A step = one frame through
  nerfies_b200.evaluation.render_frame; the collective's time is reported.
  Returns the JSON line (rank 0) or None; dump_dir receives the last frame."""
  import numpy as np
  import torch
  import torch.distributed as dist
  import nerfies_b200 as nb
  from nerfies_b200 import evaluation
  dev, world, rank = ctx['dev'], ctx['world'], ctx['rank']
  w, h = wl['frame']
  evals = 2 * wl['nc'] + wl['nf']
  max_rays = 32768
  model, params = nb.construct_nerf(0, model_config(wl), max_rays, range(N_IDS), range(2),
                                    range(N_IDS), NEAR, FAR, precision=precision, device=dev)
  cpu = lambda t: ({k: cpu(v) for k, v in t.items()} if isinstance(t, dict) else t.cpu())
  gpu = lambda t: ({k: gpu(v) for k, v in t.items()} if isinstance(t, dict) else t.to(dev))
  params_cpu = trained_like(cpu(params), seed=1)
  params = gpu(params_cpu)
  th = 0.2
  R = np.array([[np.cos(th), 0, np.sin(th)], [0, 1, 0], [-np.sin(th), 0, np.cos(th)]], np.float32)
  cam = nb.camera.Camera(orientation=R, position=[0.05, -0.02, -0.35], focal_length=1500.0,
                         principal_point=[w / 2, h / 2], image_size=[w, h],
                         radial_distortion=[0.02, -0.01, 0.0], tangential_distortion=[1e-3, -5e-4])
  md = {'warp': 17, 'appearance': 23}
  extra = {'alpha': float(wl['fw']), 'time_alpha': 0.0}

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  frame = evaluation.render_frame(model, params, cam, extra, md, max_rays=max_rays)   # warm-up
  barrier()
  sampler = ClockSampler(ctx['local_rank'])
  sampler.start()
  launches0 = model.kernel_launches()
  tms = []
  for _ in range(steps):
    t = {}
    frame = evaluation.render_frame(model, params, cam, extra, md, max_rays=max_rays, timings=t)
    tms.append((t['render_ms'], t['gather_ms']))
  barrier()
  clocks = sampler.stop()
  launches = model.kernel_launches() - launches0
  tot = torch.tensor([sum(a + b for a, b in tms), sum(b for _, b in tms)], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(tot, op=dist.ReduceOp.MAX)
  ms = float(tot[0]) / steps
  gather_ms = float(tot[1]) / steps
  if rank != 0:
    return None
  if dump_dir:
    dump_outputs(dump_dir, flat_outputs(frame))
  value = w * h * evals / (ms * 1e-3)
  line = {
      'metric': 'ray-samples/sec (coarse+fine, device-timed)', 'value': value,
      'unit': 'ray-samples/s', 'n_gpus': world, 'steps': steps, 'warmup': 1,
      'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
      'dtype': DTYPE_NAMES[precision], 'data': 'synthetic',
      'config': {'workload': workload_text(wl, w * h), 'workload_name': 'eval-1080p',
                 'precision': precision, 'rays_per_gpu': -(-w * h // world),
                 'parallelism': f'frame rows split x{world}; one NCCL all_gather of the packed (rays, 6) result',
                 'l2': 'a frame is 2.07 M rays: every launch streams far more than L2',
                 'timing': 'CUDA events on the launch stream around each frame (ray generation + render + '
                           'all_gather), max over ranks'},
      'frame_ms': ms, 'all_gather_ms': gather_ms, 'clocks': clocks, 'gpu_launches': int(launches),
  }
  if not args.no_parity:
    # a sample of the frame's pixels against the oracle, on the rays the GPU generated
    from oracle import nerfies_oracle as O
    from nerfies_b200 import camera as camera_lib
    spec = oracle_spec(wl)
    idx = torch.linspace(0, w * h - 1, 96).round().long()
    rays = camera_lib.camera_to_rays(cam, dev)
    sub = {'origins': rays['origins'].reshape(-1, 3)[idx.to(dev)].cpu(),
           'directions': rays['directions'].reshape(-1, 3)[idx.to(dev)].cpu(),
           'metadata': {k: torch.full((96, 1), v, dtype=torch.int32) for k, v in md.items()}}
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    with torch.no_grad():
      ref = O.render_forward(params_cpu, spec, sub, warp_alpha=extra['alpha'])
    got = {k: frame[k].reshape((w * h,) + tuple(frame[k].shape[2:]))[idx.to(dev)].cpu() for k in ('rgb', 'depth', 'acc')}
    par = {f'max_rel_{k}': rel_err(got[k], ref['fine'][k]) for k in ('rgb', 'depth', 'acc')}
    par['psnr_db'] = psnr_db(got['rgb'], ref['fine']['rgb'])
    b = PARITY_BOUNDS[precision]
    par['bounds'] = {'e2e': b['e2e'], 'psnr_db': b['psnr_db']}
    par['ok'] = bool(max(par[f'max_rel_{k}'] for k in ('rgb', 'depth', 'acc')) < b['e2e'] and par['psnr_db'] > b['psnr_db'])
    par['pixels'] = 96
    line['parity'] = par
  return line


def measure_train_step(args, wl, ctx):
  """--workload quarterhd-trainstep (SURVEY §8(f) #1): a step = nerfies_b200.training.train_step
  (value_and_grad + gradient all-reduce + Adam).  The global batch is fixed (the reference's
  6144 rays) and split over the ranks."""
  import torch
  import torch.distributed as dist
  import nerfies_b200 as nb
  from nerfies_b200 import training
  dev, world, rank = ctx['dev'], ctx['world'], ctx['rank']
  B = max(1, (args.rays or wl['rays']) // world)
  evals = 2 * wl['nc'] + wl['nf']
  model, params = nb.construct_nerf(0, model_config(wl), B, range(N_IDS), range(2), range(N_IDS), NEAR, FAR,
                                    precision='fp32', device=dev)
  cpu = lambda t: ({k: cpu(v) for k, v in t.items()} if isinstance(t, dict) else t.cpu())
  gpu = lambda t: ({k: gpu(v) for k, v in t.items()} if isinstance(t, dict) else t.to(dev))
  state = training.create_train_state(model, gpu(trained_like(cpu(params), seed=1)), warp_alpha=float(wl['fw']))
  rays = synthetic_rays(B, 1000 + rank, wl)
  g = torch.Generator().manual_seed(77 + rank)
  batch = {'origins': rays['origins'].to(dev), 'directions': rays['directions'].to(dev),
           'metadata': {k: v.to(dev) for k, v in rays['metadata'].items()},
           'rgb': torch.rand(B, 3, generator=g).to(dev)}
  sp = training.ScalarParams(learning_rate=1e-3)
  chunk = 1024
  kw = {}
  if wl.get('reg'):
    # gpu_vrig_paper.gin:31,52-61
    sp = training.ScalarParams(learning_rate=1e-3, elastic_loss_weight=0.001, background_loss_weight=1.0)
    batch['background_points'] = (torch.rand(B, 3, generator=g) * 0.6 - 0.3).to(dev)
    kw = dict(use_elastic_loss=True, elastic_reduce_method='weight', use_background_loss=True)
    chunk = 512

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  losses = []
  for _ in range(max(1, min(args.warmup, 2))):
    state, stats, _ = training.train_step(model, 0, state, batch, sp, chunk_rays=chunk, **kw)
  barrier()
  sampler = ClockSampler(ctx['local_rank'])
  sampler.start()
  tms = []
  launches0 = model.kernel_launches()
  barrier()
  for _ in range(args.steps):
    t = {}
    state, stats, _ = training.train_step(model, 0, state, batch, sp, chunk_rays=chunk, timings=t, **kw)
    tms.append(t)
    losses.append(float(stats['fine']['loss/total']))
  barrier()
  clocks = sampler.stop()
  launches = model.kernel_launches() - launches0
  keys = ('value_and_grad_ms', 'all_reduce_ms', 'adam_ms')
  tot = torch.tensor([sum(sum(t[k] for k in keys) for t in tms)] + [sum(t[k] for t in tms) for k in keys],
                     device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(tot, op=dist.ReduceOp.MAX)
  if rank != 0:
    return None
  if args.dump_outputs:
    opt = state.optimizer
    dump_outputs(args.dump_outputs, {'params': opt.flat, 'adam_m': opt.m, 'adam_v': opt.v,
                                     **flat_outputs(stats)})
  ms = float(tot[0]) / args.steps
  n_params = state.optimizer.flat.numel()
  return {
      'metric': 'ray-samples/sec (coarse+fine, device-timed)', 'value': world * B * evals / (ms * 1e-3),
      'unit': 'ray-samples/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(1, min(args.warmup, 2)),
      'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
      'dtype': 'fp32 (training tier: layer-wise SIMT GEMMs, forward + backward)', 'data': 'synthetic',
      'config': {'workload': workload_text(wl, B), 'workload_name': args.workload,
                 'rays_per_gpu': B, 'global_batch': B * world, 'precision': 'fp32',
                 'parallelism': f'data parallel x{world}: one NCCL all_reduce of the flat gradient '
                                f'({n_params} fp32 = {n_params * 4 / 1e6:.1f} MB) per step',
                 'timing': 'CUDA events on the launch stream around the three phases of a step, max over ranks'},
      'value_and_grad_ms': float(tot[1]) / args.steps, 'all_reduce_ms': float(tot[2]) / args.steps,
      'adam_ms': float(tot[3]) / args.steps, 'train_flop_per_step': 3 * world * B * evals * wl['flop'],
      'achieved_tflops_fp32': 3 * world * B * evals * wl['flop'] / (ms * 1e-3) / 1e12 / world,
      'loss_first_last': [losses[0], losses[-1]], 'clocks': clocks, 'gpu_launches': int(launches),
      'stats_last_step': {lv: {k: float(v) for k, v in stats[lv].items()} for lv in ('coarse', 'fine')},
  }


def run_b200(args):
  import torch
  import torch.distributed as dist

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  if world > 1:
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
  if args.gpus != world and rank == 0 and world > 1:
    print(f'warning: --gpus {args.gpus} but WORLD_SIZE={world}', file=sys.stderr)
  torch.cuda.set_device(local_rank)
  dev = torch.device('cuda', local_rank)
  wl = WORKLOADS[args.workload]
  precision = args.precision or 'fp16x3'
  total_rays = args.rays or wl['rays']
  B = total_rays if args.scaling == 'weak' else max(1, total_rays // world)
  evals = 2 * wl['nc'] + wl['nf']
  ctx = {'dev': dev, 'world': world, 'rank': rank, 'local_rank': local_rank,
         'flush': torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)}

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  if wl.get('trainstep'):
    line = measure_train_step(args, wl, ctx)
    if rank == 0:
      emit(line)
    if world > 1:
      dist.destroy_process_group()
    return
  if 'frame' in wl:
    line = measure_eval_frame(args, wl, precision, ctx, args.steps, dump_dir=args.dump_outputs)
    if rank == 0:
      emit(line)
    if world > 1:
      dist.destroy_process_group()
    return
  main = measure(precision, wl, B, args, ctx, want_parity=not args.no_parity)
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, flat_outputs(main['out']))

  # End to end through the C ABI's host entry point: host buffers in, host
  # buffers out, H2D + D2H inside the timed region.
  model, variables, rays_host = main['model'], main['variables'], main['rays_host']
  host_rays = {'origins': rays_host['origins'].numpy(),
               'directions': rays_host['directions'].numpy(),
               'metadata': {k: v.numpy() for k, v in rays_host['metadata'].items()}}
  model.apply_host(variables, host_rays, warp_extra=main['warp_extra'])   # warm-up
  e2e_steps = max(2, min(args.steps, 5))
  barrier()
  t0 = time.perf_counter()
  for _ in range(e2e_steps):
    model.apply_host(variables, host_rays, warp_extra=main['warp_extra'])
  barrier()
  e2e_s = torch.tensor([(time.perf_counter() - t0) / e2e_steps], device=dev,
                       dtype=torch.float64)
  if world > 1:
    dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
  e2e_value = world * B * evals / float(e2e_s)
  n_id_arrays = 1 + int(wl['app']) + int(wl['cam'])
  h2d = B * (12 + 12 + 4 * n_id_arrays)   # origins, directions, metadata ids
  d2h = B * 2 * 6 * 4                     # (B,6) per level

  also = {}
  if not args.no_also:
    for other in ('bf16',):
      if other == precision:
        continue
      r = measure(other, wl, B, args, ctx, want_parity=not args.no_parity)
      also[other] = r
    if world > 1 and args.scaling == 'weak':
      # strong scaling beside the weak headline: the same TOTAL batch split over the ranks
      r = measure(precision, wl, max(1, total_rays // world), args, ctx, want_parity=False)
      also['strong'] = r
    if args.workload == 'northstar':
      # BASELINE.json's eval config rides along (one warm-up + one timed 1080p frame), so that the
      # driver's 1 -> 8 GPU runs record the frame-time curve too; never allowed to break the line
      try:
        ev = measure_eval_frame(args, WORKLOADS['eval-1080p'], precision, ctx, 1)
        if ev is not None:
          also['eval_1080p'] = {k: ev[k] for k in ('value', 'frame_ms', 'all_gather_ms', 'n_gpus', 'parity')
                                if k in ev}
          also['eval_1080p']['workload'] = ev['config']['workload']
      except Exception as e:   # pylint: disable=broad-except
        also['eval_1080p'] = {'error': repr(e)}

  if rank != 0:
    if world > 1:
      dist.destroy_process_group()
    return

  peaks = {}
  try:
    with open(os.path.join(REPO, 'MEASURED_PEAKS.json')) as f:
      peaks = json.load(f)
  except OSError:
    pass
  line = {
      'metric': 'ray-samples/sec (coarse+fine, device-timed)',
      'value': main['value'], 'unit': 'ray-samples/s', 'n_gpus': world,
      'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': main['ms_per_step'],
      'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
      'dtype': DTYPE_NAMES[precision],
      'data': 'synthetic',
      'config': {
          'workload': workload_text(wl, B),
          'workload_name': args.workload,
          'rays_per_gpu': B, 'precision': precision,
          'parallelism': f'ray sharding x{world}, no data-path collective',
          'l2': 'L2 flushed (256 MiB memset) between timed iterations; the per-step working set '
                '(per-sample outputs) also exceeds L2 at the default batch',
          'timing': 'per-step CUDA events on the launch stream, summed, max over ranks',
      },
      'clocks': main['clocks'],
      'e2e': {'value': e2e_value, 'unit': 'ray-samples/s',
              'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
              'api': 'NerfModel.apply_host -> nfb_render_forward_host (host '
                     'buffers, pinned staging, H2D+D2H timed)'},
      'gpu_launches': main['launches'],
      'roofline': roofline(main, wl, B, peaks, precision),
      'wall_s_timed_region': main['wall'],
  }
  if 'parity' in main:
    line['parity'] = main['parity']
  if also:
    line['also'] = {}
    for name, r in also.items():
      if name == 'eval_1080p':
        line['also'][name] = r
      elif name == 'strong':
        b2 = max(1, total_rays // world)
        line['also']['strong_scaling'] = {
            'precision': precision, 'total_rays': b2 * world, 'rays_per_gpu': b2,
            'value': r['value'], 'ms_per_step': r['ms_per_step'],
            'note': 'same workload with the TOTAL batch fixed and split over the ranks; '
                    'efficiency = value / (N x the N=1 value of the default line)'}
      else:
        line['also'][name] = {
            'value': r['value'], 'ms_per_step': r['ms_per_step'],
            'dtype': DTYPE_NAMES[name], 'roofline_frac': roofline(r, wl, B, peaks, name)['frac'],
            'fine_kernel_ms': r['field_ms'][1], 'clocks': r['clocks'],
            'parity': r.get('parity')}
  if not args.no_cpu_baseline and world == 1:      # rank 0 at N = 1 only (task contract)
    line['cpu_baseline'] = cpu_baseline(args.cpu_seconds, args.workload)
  bad = 'parity' in line and not line['parity']['ok']
  if bad:
    line['invalid'] = 'parity check failed: errors exceed the stated bound of this precision mode'
  emit(line)
  if world > 1:
    dist.destroy_process_group()
  if bad:
    sys.exit(3)


_SAVED_STDOUT = None


def quiet_stdout():
  """Route fd 1 to stderr until emit(): libraries (NCCL's version banner, ...)
  must not print in front of the one JSON line the driver parses."""
  global _SAVED_STDOUT
  sys.stdout.flush()
  _SAVED_STDOUT = os.dup(1)
  os.dup2(2, 1)


def emit(line):
  sys.stdout.flush()
  if _SAVED_STDOUT is not None:
    os.dup2(_SAVED_STDOUT, 1)
  print(json.dumps(line), flush=True)


def main():
  args = parse_args()
  quiet_stdout()
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_b200(args)


if __name__ == '__main__':
  main()
