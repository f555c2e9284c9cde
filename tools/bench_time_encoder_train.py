"""Cost of training the 'time' / 'blend' warp metadata encoders (the TimeEncoder backward).

Times training.value_and_grad at the quarterhd-trainstep size of bench.py (6,144 rays x (128+128)
samples, gpu_quarterhd.gin model dimensions, fp32 training tier) for two pairs of models that
differ only in the warp metadata encoder:
  se3:         'glo' vs 'time'  (metadata['time'] per ray, time_alpha = F / 2: half-open window)
  translation: 'glo' vs 'blend' (time_alpha = 0.5)
The two models of a pair alternate in one process after a warm-up; every call is timed with CUDA
events on the launch stream.  Prints one JSON line with the GPU's name and power limit.

  python tools/bench_time_encoder_train.py [--rounds 8] [--warmup 2]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
  sys.path.insert(0, REPO)

import bench  # noqa: E402  (workload dimensions, trained-like weights, synthetic rays)

PAIRS = (('se3', 'glo', 'time'), ('translation', 'glo', 'blend'))


def gpu_info(index):
  out = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit,clocks.max.sm',
                        '--format=csv,noheader'], capture_output=True, text=True, check=True).stdout.strip()
  name, power, clock = [s.strip() for s in out.split(',')]
  return {'name': name, 'power_limit': power, 'max_sm_clock': clock}


def make(field, enc, wl, B, dev):
  import dataclasses
  import torch
  import nerfies_b200 as nb
  from nerfies_b200 import training
  cfg = dataclasses.replace(bench.model_config(wl), warp_field_type=field, warp_metadata_encoder_type=enc)
  model, params = nb.construct_nerf(0, cfg, B, range(bench.N_IDS), range(2), range(bench.N_IDS), bench.NEAR,
                                    bench.FAR, precision='fp32', device=dev)
  cpu = lambda t: ({k: cpu(v) for k, v in t.items()} if isinstance(t, dict) else t.cpu())
  gpu = lambda t: ({k: gpu(v) for k, v in t.items()} if isinstance(t, dict) else t.to(dev))
  params = gpu(bench.trained_like(cpu(params), seed=1))
  rays = bench.synthetic_rays(B, 1000, wl)
  g = torch.Generator().manual_seed(77)
  md = {k: v.to(dev) for k, v in rays['metadata'].items()}
  md['time'] = (torch.rand(B, 1, generator=g) * 2 - 1).to(dev)       # the 'time' encoder's input
  batch = {'origins': rays['origins'].to(dev), 'directions': rays['directions'].to(dev), 'metadata': md,
           'rgb': torch.rand(B, 3, generator=g).to(dev)}
  extra = {'alpha': float(wl['fw']),
           'time_alpha': 0.5 if enc == 'blend' else 0.5 * model.metadata_encoder_num_freqs}
  grads = torch.zeros(sum(r * c for _, r, c in model.handle(B).param_specs), device=dev)

  def step():
    grads.zero_()
    return training.value_and_grad(model, params, batch, extra, chunk_rays=1024, grads=grads)
  return step


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--rounds', type=int, default=8)
  ap.add_argument('--warmup', type=int, default=2)
  args = ap.parse_args()
  import torch
  assert torch.cuda.is_available(), 'needs a CUDA device'
  dev = torch.device('cuda', 0)
  torch.cuda.set_device(dev)
  wl = bench.WORKLOADS['quarterhd-trainstep']
  B = wl['rays']
  result = {'metric': 'training.value_and_grad ms per call (device events)', 'gpu': gpu_info(0),
            'workload': f'training.value_and_grad, photometric loss: {B} rays x ({wl["nc"]}+{wl["nf"]}) samples, '
                        'gpu_quarterhd.gin model dims, fp32 training tier, chunk_rays 1024, trained-like random '
                        'weights, TimeEncoder metadata_encoder_num_freqs 1',
            'rounds': args.rounds, 'warmup': args.warmup, 'pairs': {}}
  for field, base, enc in PAIRS:
    steps = {base: make(field, base, wl, B, dev), enc: make(field, enc, wl, B, dev)}
    for _ in range(args.warmup):
      for f in steps.values():
        f()
    torch.cuda.synchronize()
    ms = {k: [] for k in steps}
    for _ in range(args.rounds):
      for k, f in steps.items():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        f()
        ev[1].record()
        ev[1].synchronize()
        ms[k].append(ev[0].elapsed_time(ev[1]))
    ratios = [b / a - 1.0 for a, b in zip(ms[base], ms[enc])]
    result['pairs'][f'{field}:{base}-vs-{enc}'] = {
        'ms_' + k: {'median': statistics.median(v), 'min': min(v), 'max': max(v)} for k, v in ms.items()}
    result['pairs'][f'{field}:{base}-vs-{enc}']['overhead_median_of_paired_rounds'] = statistics.median(ratios)
    result['pairs'][f'{field}:{base}-vs-{enc}']['overhead_per_round'] = ratios
  print(json.dumps(result))


if __name__ == '__main__':
  main()
