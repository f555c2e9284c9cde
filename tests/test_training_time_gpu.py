"""Training with the 'time' and 'blend' warp metadata encoders (modules.TimeEncoder,
warping.py:98-148, 309-320): gradients of the photometric loss and of the regularisers
against torch.autograd on the oracle in float64, the blend endpoints, the warp Jacobian, and
train_step end to end.

Tolerances as in test_training_gpu.py: 5e-3 of each tensor's largest gradient entry for the
shared and coarse-level parameters (the TimeEncoder and the GLO tables are shared), 2e-2 for
nerf_mlps_fine, whose z the CUDA run resamples from its own fp32 coarse weights.
"""
import numpy as np
import pytest
import torch

from oracle import nerfies_oracle as O
from tests.golden_util import Golden, flatten, model_from_spec, rel_err, tree_to_device

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _params64(g):
  def conv(t):
    return {k: conv(v) for k, v in t.items()} if isinstance(t, dict) else t.double().clone()
  return conv(g.params)


def _warp_meta(g):
  """The warp field's metadata of the ray batch (models.py:252-254)."""
  md = g.rays['metadata']
  return md['time'] if g.spec.warp_metadata_encoder_type == 'time' else md['warp']


def _is_time_encoder(k):
  return k.startswith('warp_field/') and '/mlp/' in k and ('metadata_encoder' in k or 'time_encoder' in k)


def _is_glo(k):
  return k.endswith('/embed/embedding') and k.startswith('warp_field/')


def _oracle(g, p64, target, time_alpha, zc, zf, sp=None, elastic=False, reduce='median', etype='log_svals',
            warp_reg=False, bg=None):
  """training.py:171-212, 246-257 on the oracle in float64, both levels on the given z, every
  metadata encoding with `time_alpha`.  Returns (loss terms, gradients)."""
  spec = g.spec
  leaves = flatten(p64)
  for v in leaves.values():
    v.requires_grad_(True)
  total, parts = 0.0, {}
  for lv, z in (('coarse', zc), ('fine', zf)):
    out = O.render_level(p64, spec, lv, g.rays, z, g.warp_alpha, dtype=torch.float64, time_alpha=time_alpha)
    parts['rgb_' + lv] = ((out['rgb'] - target.double())**2).mean()
    total = total + parts['rgb_' + lv]
    weights = out['weights'].detach()                               # lax.stop_gradient
    if elastic and lv == 'coarse':                                  # training.py:176-193, 242-244
      B, S = weights.shape
      meta = _warp_meta(g)[:, None, :].expand(B, S, 1)
      pts = out['points']
      if reduce == 'median':
        idx = O.compute_depth_index(weights)
        pts = torch.gather(pts, 1, idx[:, None, None].expand(B, 1, 3))
        meta = meta[:, :1]
      jac = O.warp_jacobian(p64['warp_field'], spec, pts, meta, g.warp_alpha, time_alpha=time_alpha,
                            create_graph=True)
      loss, _ = O.compute_elastic_loss(jac, loss_type=etype)
      if reduce == 'weight':
        loss = weights * loss
      parts['elastic'] = loss.sum(dim=-1).mean()
      total = total + sp.elastic_loss_weight * parts['elastic']
    if warp_reg:                                                    # training.py:194-207 (no metadata)
      r = O.level_regularisers(p64, spec, out, g.rays, g.warp_alpha, use_warp_reg_loss=True,
                               warp_reg_loss_alpha=sp.warp_reg_loss_alpha,
                               warp_reg_loss_scale=sp.warp_reg_loss_scale)
      parts['warp_reg_' + lv] = r['loss/warp_reg']
      total = total + sp.warp_reg_loss_weight * r['loss/warp_reg']
  if bg is not None:
    l = O.compute_background_loss(p64, spec, bg['points'].double(), bg['ids'], bg['noise'].double(),
                                  g.warp_alpha, time_alpha=time_alpha).mean()
    parts['background'] = l
    total = total + sp.background_loss_weight * l
  total.backward()
  grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in leaves.items()}
  return {k: float(v.detach()) for k, v in parts.items()}, grads


def _oracle_z(g, time_alpha):
  with torch.no_grad():
    fwd = O.render_forward(_params64(g), g.spec, g.rays, warp_alpha=g.warp_alpha, dtype=torch.float64,
                           t_rand=g.t_rand, u_rand=g.u_rand, time_alpha=time_alpha)
  return fwd['coarse']['z_vals'], fwd['fine']['z_vals']


def _background(g, n=23):
  gen = torch.Generator().manual_seed(3)
  return dict(points=torch.rand(n, 3, generator=gen) * 0.5 - 0.25,
              ids=torch.randint(0, g.spec.num_warp_embeddings, (n, 1), generator=gen),
              noise=0.001 * torch.randn(n, 3, generator=gen))


def _cuda(g, target, time_alpha, reg=None, model=None):
  from nerfies_b200 import training
  model = model or model_from_spec(g.spec_dict, device=DEV)
  if isinstance(reg, dict):
    reg = training.make_reg(model, **reg)
  losses, grads = training.value_and_grad(model, tree_to_device(g.params, DEV), dict(g.rays, rgb=target),
                                          {'alpha': g.warp_alpha, 'time_alpha': time_alpha}, chunk_rays=5,
                                          t_rand=g.t_rand, u_rand=g.u_rand, reg=reg)
  torch.cuda.synchronize()
  return {k: float(v) for k, v in losses.items()}, flatten(training.grads_to_tree(model, grads))


def _worst(got, ref):
  worst = {}
  for k, r in ref.items():
    a = got[k].cpu().double().reshape(r.shape)
    worst[k] = float((a - r).abs().max()) / (float(r.abs().max()) + 1e-12)
  return {k: v for k, v in worst.items() if v > (2e-2 if 'nerf_mlps_fine' in k else 5e-3)}


@pytest.mark.parametrize('name,time_alpha', [('time_small', None), ('blend_small', 0.35), ('blend_small', 1.0)],
                         ids=['time_small', 'blend_small-0.35', 'blend_small-1.0'])
def test_time_encoder_gradients_match_autograd_on_the_oracle(name, time_alpha):
  g = Golden(name)
  ta = g.time_alpha if time_alpha is None else time_alpha       # time_small: 1.6, the window is half open
  torch.manual_seed(21)
  target = torch.rand(g.rays['origins'].shape[0], 3)
  zc, zf = _oracle_z(g, ta)
  parts, ref = _oracle(g, _params64(g), target, ta, zc, zf)
  # the check must be able to fail: every TimeEncoder leaf has a reference gradient far from zero
  # (a missing or zero gradient is off by 100 % of the tensor's largest entry)
  tk = [k for k in ref if _is_time_encoder(k)]
  assert len(tk) == 14 and min(float(ref[k].abs().max()) for k in tk) > 1e-8
  assert min(float(ref[k].abs().max()) for k in tk if '/logit/' in k) > 1e-5
  losses, got = _cuda(g, target, ta)
  assert abs(losses['coarse'] - parts['rgb_coarse']) < 1e-5 * max(1.0, parts['rgb_coarse'])
  bad = _worst(got, ref)
  assert not bad, bad


@pytest.mark.parametrize('time_alpha', [0.0, 1.0])
def test_blend_endpoints(time_alpha):
  """(1 - time_alpha) glo + time_alpha time (warping.py:132-133): at time_alpha = 0 the TimeEncoder
  gets no gradient, from the rays or from the background points; at 1 the GLO table gets none."""
  from nerfies_b200 import training
  g = Golden('blend_small')
  torch.manual_seed(22)
  target = torch.rand(g.rays['origins'].shape[0], 3)
  sp = training.ScalarParams(learning_rate=1e-3, background_loss_weight=60.0)
  bg = _background(g)
  zc, zf = _oracle_z(g, time_alpha)
  _, ref = _oracle(g, _params64(g), target, time_alpha, zc, zf, sp=sp, bg=bg)
  reg = dict(scalar_params=sp, use_background_loss=True, background_points=bg['points'],
             background_warp_ids=bg['ids'], background_noise=bg['noise'])
  _, got = _cuda(g, target, time_alpha, reg=reg)
  zero = _is_time_encoder if time_alpha == 0.0 else _is_glo
  other = _is_glo if time_alpha == 0.0 else _is_time_encoder
  zk = [k for k in got if zero(k)]
  assert zk and all(float(got[k].abs().max()) == 0.0 for k in zk), zk
  assert max(float(got[k].abs().max()) for k in got if other(k)) > 1e-6
  bad = _worst(got, ref)
  assert not bad, bad


@pytest.mark.parametrize('case', [
    dict(name='time_small', elastic=True, reduce='median', etype='log_svals'),
    dict(name='time_small', elastic=True, reduce='weight', etype='log_svals'),
    dict(name='time_small', warp_reg=True),
    dict(name='time_small', background=True),
    dict(name='blend_small', elastic=True, reduce='median', etype='jtj'),
    dict(name='blend_small', background=True),
], ids=lambda c: '-'.join(f'{k}={v}' for k, v in c.items()))
def test_time_encoder_regulariser_gradients_match_autograd_on_the_oracle(case):
  """The regularisers of train_step with the 'time' / 'blend' encoders, weights as in
  test_regulariser_gradients_match_autograd_on_the_oracle.  The background points carry integer
  ids for every encoder: the 'time' encoder sees float(id) (training.py:121-131)."""
  from nerfies_b200 import training
  g = Golden(case['name'])
  ta = g.time_alpha
  torch.manual_seed(11)
  target = torch.rand(g.rays['origins'].shape[0], 3)
  sp = training.ScalarParams(learning_rate=1e-3, elastic_loss_weight=5.0, warp_reg_loss_weight=3.0,
                             warp_reg_loss_alpha=-2.0, warp_reg_loss_scale=0.05, background_loss_weight=60.0)
  zc, zf = _oracle_z(g, ta)
  bg = _background(g) if case.get('background') else None
  kw = dict(elastic=case.get('elastic', False), reduce=case.get('reduce', 'median'),
            etype=case.get('etype', 'log_svals'), warp_reg=case.get('warp_reg', False))
  parts, ref = _oracle(g, _params64(g), target, ta, zc, zf, sp=sp, bg=bg, **kw)
  _, plain = _oracle(g, _params64(g), target, ta, zc, zf)
  moved = max(float((ref[k] - plain[k]).abs().max()) / (float(ref[k].abs().max()) + 1e-12)
              for k in ref if k.startswith('warp_field/'))
  assert moved > 0.25, moved
  reg = dict(scalar_params=sp, use_elastic_loss=kw['elastic'], elastic_reduce_method=kw['reduce'],
             elastic_loss_type=kw['etype'], use_background_loss=bg is not None, use_warp_reg_loss=kw['warp_reg'])
  if bg is not None:
    reg.update(background_points=bg['points'], background_warp_ids=bg['ids'], background_noise=bg['noise'])
  losses, got = _cuda(g, target, ta, reg=reg)
  for k in ('elastic', 'warp_reg_coarse', 'background'):
    if k in parts:
      assert abs(losses[k] - parts[k]) < 2e-4 * max(abs(parts[k]), 1e-3), (k, losses[k], parts[k])
  bad = _worst(got, ref)
  assert not bad, bad


@pytest.mark.parametrize('name', ['time_small', 'blend_small'])
def test_time_encoder_warp_jacobian_matches_the_oracle(name):
  """jax.jacfwd(self.warp) (warping.py:385-387) with the TimeEncoder's embedding as a constant input,
  through warp_field.apply(return_jacobian=True) and model.apply(return_warp_jacobian=True)."""
  g = Golden(name)
  ta = g.time_alpha
  extra = {'alpha': g.warp_alpha, 'time_alpha': ta}
  model = model_from_spec(g.spec_dict, device=DEV)
  params = tree_to_device(g.params, DEV)
  p64 = O.tree_to(g.params, torch.float64)
  gen = torch.Generator().manual_seed(5)
  P = 37
  pts = torch.rand(P, 3, generator=gen) * 0.6 - 0.3
  if g.spec.warp_metadata_encoder_type == 'time':
    meta = torch.rand(P, 1, generator=gen) * 2.0 - 1.0
  else:
    meta = torch.randint(0, g.spec.num_warp_embeddings, (P, 1), generator=gen)
  wf = model.create_warp_field(model, num_batch_dims=1)
  out = wf.apply({'params': params['warp_field']}, pts, meta, extra, return_jacobian=True)
  torch.cuda.synchronize()
  ref = O.warp_jacobian(p64['warp_field'], g.spec, pts.double(), meta, g.warp_alpha, time_alpha=ta).detach()
  err = float((out['jacobian'].cpu().double() - ref).abs().max())
  assert err < 2e-5 * max(1.0, float(ref.abs().max())), err
  o2 = model.apply({'params': params}, g.rays, warp_extra=extra, return_warp_jacobian=True, return_points=True,
                   t_rand=g.t_rand, u_rand=g.u_rand)
  torch.cuda.synchronize()
  for lv in ('coarse', 'fine'):
    J = o2[lv]['warp_jacobian'].cpu()
    B, S = J.shape[:2]
    meta_bs = _warp_meta(g)[:, None, :].expand(B, S, 1).reshape(-1, 1)
    ref = O.warp_jacobian(p64['warp_field'], g.spec, o2[lv]['points'].cpu().double().reshape(-1, 3), meta_bs,
                          g.warp_alpha, time_alpha=ta).detach().reshape(B, S, 3, 3)
    assert float((J.double() - ref).abs().max()) < 2e-5 * max(1.0, float(ref.abs().max())), lv


def test_train_step_with_a_rising_time_alpha():
  """train_step on the 'blend' encoder while time_alpha moves from the GLO code to the TimeEncoder
  (the schedule the reference's driver runs, train.py:284-285)."""
  from nerfies_b200 import training
  g = Golden('blend_small')
  torch.manual_seed(23)
  B = g.rays['origins'].shape[0]
  target = torch.rand(B, 3)
  model = model_from_spec(g.spec_dict, device=DEV)
  state = training.create_train_state(model, tree_to_device(g.params, DEV), warp_alpha=g.warp_alpha)
  tree = flatten(state.optimizer.target['model'])
  time_keys = [k for k in tree if _is_time_encoder(k)]
  before = {k: tree[k].clone() for k in time_keys}
  batch = dict(g.rays, rgb=target, background_points=torch.rand(40, 3) * 0.4 - 0.2)
  sp = training.ScalarParams(learning_rate=2e-3, background_loss_weight=1.0)
  first = last = None
  for it in range(12):
    state.time_alpha = it / 11.0
    state, stats, _ = training.train_step(model, it, state, batch, sp, use_background_loss=True, chunk_rays=6)
    assert all(np.isfinite(float(v)) for lv in ('coarse', 'fine') for v in stats[lv].values())
    assert np.isfinite(float(stats['background_loss']))
    tot = float(stats['coarse']['loss/total']) + float(stats['fine']['loss/total'])
    first = tot if first is None else first
    last = tot
  assert last < 0.9 * first, (first, last)
  moved = max(float((tree[k] - before[k]).abs().max()) for k in time_keys)
  assert moved > 1e-4, moved
  # the forward path renders with the trained parameters, TimeEncoder included (the last Adam update
  # rewrote the flat vector in place, behind torch's back: re-upload)
  params = state.optimizer.target['model']
  model.invalidate_params()
  out = model.apply({'params': params}, g.rays, warp_extra=state.warp_extra)
  torch.cuda.synchronize()
  ref = O.render_forward(O.tree_to(_to_cpu(params), torch.float64), g.spec, g.rays, warp_alpha=g.warp_alpha,
                         dtype=torch.float64, time_alpha=state.time_alpha)
  err = rel_err(out['coarse']['rgb'].cpu(), ref['coarse']['rgb'])
  assert err < 1e-4, err


def _to_cpu(t):
  return {k: _to_cpu(v) for k, v in t.items()} if isinstance(t, dict) else t.detach().cpu()
