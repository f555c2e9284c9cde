"""Edge cases of the C-ABI / Python surface on the GPU: empty and single-ray
batches, batches beyond the handle's capacity, ragged render_image chunking,
parameter updates, viewdirs override, both precisions."""
import numpy as np
import pytest
import torch

from oracle import nerfies_oracle as O
from tests.golden_util import (Golden, model_from_spec, rel_err, spec_to_dict,
                               tree_to_device)

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _rays(n, spec, seed):
  r = O.synthetic_rays(n, spec, seed=seed)
  return {'origins': r['origins'].to(DEV), 'directions': r['directions'].to(DEV),
          'metadata': {k: v.to(DEV) for k, v in r['metadata'].items()}}


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'fp16x3'])
def test_empty_and_single_ray(precision):
  spec = O.OracleSpec(num_coarse_samples=128, num_fine_samples=128, near=0.02,
                      far=0.83, num_nerf_point_freqs=8,
                      sigma_activation='softplus', use_warp=True,
                      use_appearance_metadata=True, num_warp_embeddings=9,
                      num_appearance_embeddings=9)
  p = tree_to_device(O.make_trained_like(O.init_params(spec, 1)), DEV)
  model = model_from_spec(spec_to_dict(spec), precision=precision, device=DEV,
                          batch_size=8)
  rays = _rays(5, spec, 2)
  full = model.apply({'params': p}, rays, warp_extra={'alpha': 8.0})
  empty = {'origins': rays['origins'][:0], 'directions': rays['directions'][:0],
           'metadata': {k: v[:0] for k, v in rays['metadata'].items()}}
  out = model.apply({'params': p}, empty, warp_extra={'alpha': 8.0})
  assert out['fine']['rgb'].shape == (0, 3) and out['coarse']['acc'].shape == (0,)
  one = {'origins': rays['origins'][3:4], 'directions': rays['directions'][3:4],
         'metadata': {k: v[3:4] for k, v in rays['metadata'].items()}}
  out1 = model.apply({'params': p}, one, warp_extra={'alpha': 8.0})
  torch.cuda.synchronize()
  for k in ('rgb', 'depth', 'med_depth', 'acc'):
    assert torch.equal(out1['fine'][k], full['fine'][k][3:4]), k


def test_batch_larger_than_construct_batch_size_grows_the_handle():
  g = Golden('se3_small')
  model = model_from_spec(g.spec_dict, device=DEV, batch_size=4)
  p = tree_to_device(g.params, DEV)
  out = model.apply({'params': p}, g.rays, warp_extra={'alpha': g.warp_alpha})
  torch.cuda.synchronize()
  assert out['fine']['rgb'].shape[0] == g.rays['origins'].shape[0] > 4
  assert rel_err(out['coarse']['rgb'].cpu(), g.out['coarse']['rgb']) < 1e-4


def test_parameter_update_is_picked_up():
  g = Golden('se3_small')
  model = model_from_spec(g.spec_dict, device=DEV)
  p = tree_to_device(g.params, DEV)
  a = model.apply({'params': p}, g.rays, warp_extra={'alpha': g.warp_alpha})
  rgb_a = a['coarse']['rgb'].clone()
  p['nerf_mlps_coarse']['MLP_1']['logit']['bias'].add_(0.5)      # in-place update
  b = model.apply({'params': p}, g.rays, warp_extra={'alpha': g.warp_alpha})
  torch.cuda.synchronize()
  assert float((b['coarse']['rgb'] - rgb_a).abs().max()) > 1e-3
  cpu = tree_to_device(p, 'cpu')
  ref = O.render_forward(cpu, g.spec, g.rays, warp_alpha=g.warp_alpha)
  assert rel_err(b['coarse']['rgb'].cpu(), ref['coarse']['rgb']) < 1e-4


def test_viewdirs_override_and_warp_alpha_change():
  g = Golden('se3_small')
  model = model_from_spec(g.spec_dict, device=DEV)
  p = tree_to_device(g.params, DEV)
  gen = torch.Generator().manual_seed(0)
  vd = torch.randn(g.rays['origins'].shape[0], 3, generator=gen)
  vd = vd / vd.norm(dim=-1, keepdim=True)
  rays = dict(g.rays, viewdirs=vd)
  for alpha in (0.0, 1.25, 8.0):       # window closed / fractional / open
    out = model.apply({'params': p}, rays, warp_extra={'alpha': alpha})
    ref = O.render_forward(g.params, g.spec, rays, warp_alpha=alpha)
    torch.cuda.synchronize()
    for k in ('rgb', 'depth', 'acc'):
      assert rel_err(out['coarse'][k].cpu(), ref['coarse'][k]) < 1e-4, (alpha, k)


def test_render_image_ragged_chunks_match_a_single_call():
  from nerfies_b200 import evaluation
  from nerfies_b200.model_utils import Optimizer, TrainState
  g = Golden('se3_small')
  model = model_from_spec(g.spec_dict, device=DEV)
  p = tree_to_device(g.params, DEV)
  h, w = 5, 7                                   # 35 rays, chunk 8 -> 8,8,8,8,3
  spec = g.spec
  r = O.synthetic_rays(h * w, spec, seed=5)
  frame = {'origins': r['origins'].reshape(h, w, 3).to(DEV),
           'directions': r['directions'].reshape(h, w, 3).to(DEV),
           'metadata': {k: v.reshape(h, w, 1).to(DEV)
                        for k, v in r['metadata'].items()}}
  state = TrainState(Optimizer({'model': p}), warp_alpha=g.warp_alpha)
  out = evaluation.render_image(state, frame, evaluation.make_model_fn(model),
                                device_count=1, rng=0, chunk=8)
  flat = {'origins': r['origins'].to(DEV), 'directions': r['directions'].to(DEV),
          'metadata': {k: v.to(DEV) for k, v in r['metadata'].items()}}
  ref = model.apply({'params': p}, flat, warp_extra={'alpha': g.warp_alpha})
  torch.cuda.synchronize()
  assert out['rgb'].shape == (h, w, 3) and out['depth'].shape == (h, w)
  assert torch.equal(out['rgb'].reshape(-1, 3), ref['fine']['rgb'])
  assert torch.equal(out['acc'].reshape(-1), ref['fine']['acc'])


def test_coarse_only_model_and_fullhd_dims_bf16():
  # num_fine_samples = 0 (models.py:351) and the gpu_fullhd.gin dimensions.
  spec = O.OracleSpec(num_coarse_samples=64, num_fine_samples=0, near=0.1,
                      far=1.0, num_nerf_point_freqs=8, sigma_activation='softplus')
  p = O.make_trained_like(O.init_params(spec, 3))
  rays = O.synthetic_rays(10, spec, seed=4)
  model = model_from_spec(spec_to_dict(spec), device=DEV)
  out = model.apply({'params': tree_to_device(p, DEV)}, rays)
  torch.cuda.synchronize()
  assert 'fine' not in out
  ref = O.render_forward(p, spec, rays)
  assert rel_err(out['coarse']['rgb'].cpu(), ref['coarse']['rgb']) < 1e-4
  spec = O.OracleSpec(num_coarse_samples=256, num_fine_samples=256, near=0.02,
                      far=0.83, num_nerf_point_freqs=10,
                      sigma_activation='softplus', use_warp=True,
                      use_appearance_metadata=True, num_warp_embeddings=30,
                      num_appearance_embeddings=30)
  p = O.make_trained_like(O.init_params(spec, 5))
  rays = O.synthetic_rays(9, spec, seed=6)
  model = model_from_spec(spec_to_dict(spec), precision='bf16', device=DEV)
  out = model.apply({'params': tree_to_device(p, DEV)}, rays,
                    warp_extra={'alpha': 8.0})
  torch.cuda.synchronize()
  ref = O.render_forward(p, spec, rays, warp_alpha=8.0)
  mse = float(((out['fine']['rgb'].cpu() - ref['fine']['rgb'])**2).mean())
  assert -10 * np.log10(max(mse, 1e-20)) > 35


def test_protocol_error_aborts_instead_of_hanging():
  """nfb_debug_provoke_timeout makes the MMA issuer wait on an mbarrier that never completes.

  The kernel must drain (bounded spin -> host-visible abort flag -> every other
  waiter bails out) and the API must report the error, not hang the GPU."""
  import subprocess, sys, os, textwrap
  code = textwrap.dedent('''
      import torch, nerfies_b200 as nb
      cfg = nb.configs.ModelConfig(use_stratified_sampling=False, use_warp=True, warp_field_type='se3',
                                   use_appearance_metadata=True, num_coarse_samples=32, num_fine_samples=32,
                                   num_nerf_point_freqs=8, sigma_activation='softplus')
      model, params = nb.construct_nerf(0, cfg, 256, range(10), [0], range(10), near=0.02, far=0.83,
                                        precision='bf16', device='cuda:0')
      g = torch.Generator().manual_seed(0)
      rays = {'origins': torch.randn(256, 3, generator=g).cuda() * 0.1,
              'directions': torch.nn.functional.normalize(torch.randn(256, 3, generator=g), dim=-1).cuda(),
              'metadata': {'warp': torch.zeros(256, 1, dtype=torch.int32).cuda(),
                           'appearance': torch.zeros(256, 1, dtype=torch.int32).cuda()}}
      hd = model.handle(256)
      hd.lib.nfb_debug_provoke_timeout(hd.h, 1)
      try:
        model.apply({'params': params}, rays, warp_extra={'alpha': 8.0})
        torch.cuda.synchronize()
        model.apply({'params': params}, rays, warp_extra={'alpha': 8.0})
        print('NO-ERROR')
      except Exception as e:
        print('ERROR:', e)
      # the asynchronous call itself returned 0: nfb_check_abort reports the failure of submitted work,
      # nfb_reset_abort re-arms the process
      print('CHECK', hd.lib.nfb_check_abort(None, 1))
      hd.lib.nfb_debug_provoke_timeout(hd.h, 0)
      print('RESET', hd.lib.nfb_reset_abort(), hd.lib.nfb_check_abort(None, 1))
      out = model.apply({'params': params}, rays, warp_extra={'alpha': 8.0})
      torch.cuda.synchronize()
      print('RECOVERED', bool(torch.isfinite(out['fine']['rgb']).all()))
  ''')
  env = dict(os.environ)
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  out = subprocess.run([sys.executable, '-c', code], cwd=root, env=env, capture_output=True, text=True,
                       timeout=120)
  assert 'ERROR:' in out.stdout and 'mbarrier wait timed out' in out.stdout, (out.stdout, out.stderr[-2000:])
  assert 'CHECK -1' in out.stdout and 'RESET 0 0' in out.stdout and 'RECOVERED True' in out.stdout, (
      out.stdout, out.stderr[-2000:])


def test_cta_pair_variant_is_bit_identical(monkeypatch):
  """NFB_TC_PAIR=1: the experimental cta_group::2 field kernel (two CTAs share every
  weight unit, one issuer feeds both SMs) computes the same per-row arithmetic, so
  its outputs equal the default tcgen05 kernel's bit for bit - including ragged
  sizes where the follower CTA's tile lies beyond the end.  The release library reads
  no environment variables: against it, this test reruns itself in a subprocess that
  loads the -DNFB_DEV_KNOBS developer build which build() makes (through NFB_LIB_PATH)."""
  import os, subprocess, sys
  from nerfies_b200 import _lib
  if 'libnfb_dev' not in _lib.LIB_PATH:
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dev_lib = os.path.join(root, 'nerfies_b200', '_variants', 'libnfb_dev.so')
    assert os.path.exists(dev_lib), f'{dev_lib} is missing: run __graft_entry__.build()'
    out = subprocess.run(
        [sys.executable, '-m', 'pytest', '-q', '-p', 'no:cacheprovider',
         os.path.abspath(__file__) + '::test_cta_pair_variant_is_bit_identical'],
        cwd=root, env=dict(os.environ, NFB_LIB_PATH=dev_lib), capture_output=True, text=True,
        timeout=600)
    assert out.returncode == 0 and '1 passed' in out.stdout, (out.stdout[-3000:], out.stderr[-2000:])
    return
  spec = O.OracleSpec(num_coarse_samples=128, num_fine_samples=128, near=0.02, far=0.83,
                      num_nerf_point_freqs=8, sigma_activation='softplus', use_warp=True,
                      use_appearance_metadata=True, num_warp_embeddings=9,
                      num_appearance_embeddings=9)
  p = tree_to_device(O.make_trained_like(O.init_params(spec, 1)), DEV)
  model = model_from_spec(spec_to_dict(spec), precision='bf16', device=DEV, batch_size=700)
  for n in (700, 1, 3):                      # 700*128 rows = 350 pairs; tiny batches: 1 pair
    rays = _rays(n, spec, 11 + n)
    monkeypatch.delenv('NFB_TC_PAIR', raising=False)
    a = model.apply({'params': p}, rays, warp_extra={'alpha': 6.0}, return_points=True)
    torch.cuda.synchronize()
    monkeypatch.setenv('NFB_TC_PAIR', '1')
    b = model.apply({'params': p}, rays, warp_extra={'alpha': 6.0}, return_points=True)
    torch.cuda.synchronize()
    for lv in ('coarse', 'fine'):
      for k in ('rgb', 'depth', 'acc', 'warped_points'):
        assert torch.equal(a[lv][k], b[lv][k]), (n, lv, k)
  monkeypatch.delenv('NFB_TC_PAIR', raising=False)


@pytest.mark.parametrize('variant', ['default', 'white_bg_no_infinity', 'fullhd_256'])
def test_fused_composite_matches_the_staged_path(variant):
  """fp16x3: when a ray is a whole number of 128-sample tiles the field kernel finishes the
  ray on chip (volumetric rendering fused into its rgb epilogue, model_utils.py:104-136);
  otherwise - and on the return_points path - samples go through composite_kernel.  Both
  must agree to fp32 re-association, including the median depth and the two
  background / infinity variants."""
  kw = dict(num_coarse_samples=128, num_fine_samples=128)
  if variant == 'white_bg_no_infinity':
    kw.update(use_white_background=True, use_sample_at_infinity=False)
  if variant == 'fullhd_256':
    kw = dict(num_coarse_samples=256, num_fine_samples=256, num_nerf_point_freqs=10)
  spec = O.OracleSpec(near=0.02, far=0.83, sigma_activation='softplus', use_warp=True,
                      use_appearance_metadata=True, num_warp_embeddings=9,
                      num_appearance_embeddings=9, **{'num_nerf_point_freqs': 8, **kw})
  p_cpu = O.make_trained_like(O.init_params(spec, 2))
  p = tree_to_device(p_cpu, DEV)
  model = model_from_spec(spec_to_dict(spec), precision='fp16x3', device=DEV, batch_size=300)
  rays = _rays(300, spec, 21)
  fused = model.apply({'params': p}, rays, warp_extra={'alpha': 6.0}, return_weights=True)
  staged = model.apply({'params': p}, rays, warp_extra={'alpha': 6.0}, return_weights=True,
                       return_points=True)
  torch.cuda.synchronize()
  for k in ('rgb', 'depth', 'acc', 'weights'):
    assert rel_err(fused['coarse'][k].cpu(), staged['coarse'][k].cpu()) < 5e-6, k
  # median depth: identical except where the cumulative weight passes within 1e-5 of 0.5
  cum = torch.cumsum(staged['coarse']['weights'].double(), -1)
  near_half = ((cum - 0.5).abs() < 1e-5).any(-1)
  same = fused['coarse']['med_depth'] == staged['coarse']['med_depth']
  assert bool((same | near_half).all())
  # and against the oracle, end to end
  ref = O.render_forward(p_cpu, spec, {k: (v.cpu() if torch.is_tensor(v) else {a: b.cpu() for a, b in v.items()})
                                       for k, v in rays.items()}, warp_alpha=6.0)
  for k in ('rgb', 'depth', 'acc', 'weights'):
    assert rel_err(fused['coarse'][k].cpu(), ref['coarse'][k]) < 1e-4, k
  assert rel_err(fused['fine']['rgb'].cpu(), ref['fine']['rgb']) < 2e-3
