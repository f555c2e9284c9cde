"""Host logic of bench.py's CPU legs (the reference arm the driver runs beside the b200 arm)."""
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
  sys.path.insert(0, REPO)


def test_oracle_pool_two_processes():
  """Ray-sharded multi-process layout: two workers render their shards between a barrier and
  the last finish; the pool survives a second command and shuts down cleanly."""
  import bench
  pool = bench.OraclePool(2, 1, 'quarterhd-train', 128)
  try:
    assert pool.ok
    t1 = pool.run(64)
    t2 = pool.run(64)
    assert t1 and t1 > 0 and t2 and t2 > 0
  finally:
    pool.close()
  assert all(not p.is_alive() for p in pool.ps)


def test_dump_outputs_is_float_bounded_and_repeatable(tmp_path, monkeypatch):
  """--dump-outputs: nested outputs -> one float .npy per leaf; above the size bound every
  array keeps the same seeded rows, identically from run to run."""
  import numpy as np
  import torch
  import bench
  monkeypatch.setattr(bench, 'DUMP_MAX_BYTES', 4096)
  out = {'coarse': {'rgb': torch.arange(3000.).reshape(1000, 3), 'acc': torch.arange(1000.)},
         'fine': {'loss/total': torch.tensor(0.5, dtype=torch.float64), 'steps': 3}}
  flat = bench.flat_outputs(out)
  assert sorted(flat) == ['coarse_acc', 'coarse_rgb', 'fine_loss_total', 'fine_steps']
  for d in ('a', 'b'):
    bench.dump_outputs(str(tmp_path / d), flat)
  files = sorted(os.listdir(tmp_path / 'a'))
  assert files == ['coarse_acc.npy', 'coarse_rgb.npy', 'fine_loss_total.npy', 'fine_steps.npy']
  assert sum(os.path.getsize(tmp_path / 'a' / f) for f in files) <= 4096 + 4 * 128
  a = {f[:-4]: np.load(tmp_path / 'a' / f) for f in files}
  for k, v in a.items():
    assert v.dtype in (np.float32, np.float64)
    assert np.array_equal(v, np.load(tmp_path / 'b' / (k + '.npy')))
  assert 0 < a['coarse_acc'].shape[0] < 1000
  assert np.array_equal(a['coarse_rgb'][:, 0] / 3, a['coarse_acc'])   # the same rows of both
  assert a['fine_loss_total'].dtype == np.float64 and float(a['fine_steps']) == 3.0


def test_reference_line_keys(monkeypatch, capsys):
  """--impl reference prints one JSON line with the contract's keys (tiny sample)."""
  import json
  import bench

  class FakeLayout:
    def __init__(self, wl_name, max_rays):
      pass

    def sample(self, budget_s):
      return (1000.0, 4, 256, 0.1, '256 rays, one process x 4 torch threads')

    def close(self):
      pass
  monkeypatch.setattr(bench, 'CpuLayout', FakeLayout)
  monkeypatch.setattr(sys, 'argv', ['bench.py', '--impl', 'reference', '--steps', '2', '--warmup', '1'])
  monkeypatch.setenv('RANK', '0')
  args = bench.parse_args()
  bench.run_reference(args)
  line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
  for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better',
            'config', 'cpu_baseline', 'e2e'):
    assert k in line
  assert line['impl'] == 'reference' and line['e2e']['h2d_bytes_per_step'] == 0
  assert line['cpu_baseline']['cores'] == 4 and line['value'] == 1000.0
