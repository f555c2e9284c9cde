"""Mirror of the optimisation step of nerfies/training.py (SURVEY §8(f) #1).

  state = training.create_train_state(model, params)       # flat fp32 parameter / Adam buffers
  state, stats, rng = training.train_step(model, rng, state, batch, scalar_params)

`train_step` has the reference's signature (training.py:138-147) and does what its
body does (training.py:214-271): value_and_grad of the photometric loss
(mean squared error of the coarse and of the fine rgb against batch['rgb']), the
gradient mean over the devices (lax.pmean -> ONE NCCL all_reduce of the flat gradient
vector), and flax.optim.Adam's update.  Gradients come from
`nfb_train_value_and_grad` (hand-written fp32 kernels, include/nerfies_b200.h), the
update from `nfb_adam_step`; torch is the allocator and the NCCL binding.

The regularisers of train_step - the elastic loss on the warp Jacobian (training.py:71-115,
176-193), the warp regulariser (training.py:194-207) and the background loss
(training.py:118-135, 246-257) - are part of the same native call
(`nfb_train_value_and_grad_reg`, SURVEY §8(f) #2).  The reference draws the background points'
warp ids and noise with jax.random (training.py:122-126); here they come from a torch
generator seeded by `rng_key` (or are passed in the batch): same distribution, different stream.
"""
import ctypes
import dataclasses
import math
from typing import Any, Dict

import torch
import torch.distributed as dist

from nerfies_b200 import _lib
from nerfies_b200 import model_utils
from nerfies_b200.models import _prep_f32, _prep_ids, _ptr, _stream


@dataclasses.dataclass
class ScalarParams:
  """training.ScalarParams (training.py:35-43)."""
  learning_rate: float
  elastic_loss_weight: float = 0.0
  warp_reg_loss_weight: float = 0.0
  warp_reg_loss_alpha: float = -2.0
  warp_reg_loss_scale: float = 0.001
  background_loss_weight: float = 0.0
  background_noise_std: float = 0.001


class AdamOptimizer(model_utils.Optimizer):
  """flax.optim.Adam(learning_rate) wrapped like flax.optim.Optimizer: `.target` is the
  parameter pytree ({'model': params}); its leaves are views into one flat fp32 vector, so the
  update and the gradient all-reduce are single passes over contiguous memory."""

  def __init__(self, target, flat, specs, beta1=0.9, beta2=0.999, eps=1e-8):
    super().__init__(target)
    self.flat = flat
    self.specs = specs                      # [(name, offset, numel)] in nfb_param_info order
    self.m = torch.zeros_like(flat)
    self.v = torch.zeros_like(flat)
    self.step = 0
    self.beta1, self.beta2, self.eps = beta1, beta2, eps

  def apply_gradient(self, grad_flat, learning_rate):
    """optimizer.apply_gradient(grad, learning_rate=...) (training.py:268-269); in place."""
    self.step += 1
    lib = _lib.load()
    with torch.cuda.device(self.flat.device):
      _lib.check(lib.nfb_adam_step(_ptr(self.flat), _ptr(grad_flat), _ptr(self.m), _ptr(self.v),
                                   self.flat.numel(), float(learning_rate), self.beta1, self.beta2,
                                   self.eps, self.step, _stream()))
    return self


def create_train_state(model, params, warp_alpha=0.0, time_alpha=0.0):
  """Flattens the parameter pytree (Flax names) into one fp32 vector in the library's parameter
  order and rebuilds the pytree as views of it; returns model_utils.TrainState with an
  AdamOptimizer (train.py:219-221: optimizer = flax.optim.Adam(lr).create(params))."""
  hd = model.handle(1)
  specs, off = [], 0
  for name, rows, cols in hd.param_specs:
    specs.append((name, off, rows * cols))
    off += rows * cols
  flat = torch.zeros(off, device=model.device, dtype=torch.float32)
  tree: Dict[str, Any] = {}
  for (name, o, n), (_, rows, cols) in zip(specs, hd.param_specs):
    node = params
    for part in name.split('/'):
      node = node[part]
    src = torch.as_tensor(node).to(device=model.device, dtype=torch.float32)
    flat[o:o + n] = src.reshape(-1)
    view = flat[o:o + n].view(src.shape)
    t = tree
    parts = name.split('/')
    for part in parts[:-1]:
      t = t.setdefault(part, {})
    t[parts[-1]] = view
  opt = AdamOptimizer({'model': tree}, flat, specs)
  return model_utils.TrainState(opt, warp_alpha=warp_alpha, time_alpha=time_alpha)


def make_reg(model, scalar_params=None, use_elastic_loss=False, elastic_reduce_method='median',
             elastic_loss_type='log_svals', use_background_loss=False, use_warp_reg_loss=False,
             background_points=None, background_warp_ids=None, background_noise=None):
  """The regulariser switches of train_step (training.py:138-147) + ScalarParams -> nfb_train_reg.
  Returns (TrainReg, keepalive list of the device tensors it points to)."""
  sp = scalar_params
  reg = _lib.TrainReg()
  keep = []
  if elastic_loss_type not in _lib.ELASTIC_TYPES:
    raise NotImplementedError(f'elastic loss type {elastic_loss_type!r} (the reference notes that '
                              "'nr' produces NaNs, training.py:59)")
  reg.use_elastic_loss = int(bool(use_elastic_loss))
  reg.elastic_reduce_method = _lib.ELASTIC_REDUCE[elastic_reduce_method]
  reg.elastic_loss_type = _lib.ELASTIC_TYPES[elastic_loss_type]
  reg.elastic_loss_weight = float(sp.elastic_loss_weight) if sp else 0.0
  reg.use_warp_reg_loss = int(bool(use_warp_reg_loss))
  reg.warp_reg_loss_weight = float(sp.warp_reg_loss_weight) if sp else 0.0
  reg.warp_reg_loss_alpha = float(sp.warp_reg_loss_alpha) if sp else -2.0
  reg.warp_reg_loss_scale = float(sp.warp_reg_loss_scale) if sp else 0.001
  reg.use_background_loss = int(bool(use_background_loss))
  if use_background_loss:
    dev = model.device
    pts = _prep_f32(background_points, dev).reshape(-1, 3).contiguous()
    ids = _prep_ids(torch.as_tensor(background_warp_ids).reshape(pts.shape[0], -1), dev)
    noise = None if background_noise is None else _prep_f32(background_noise, dev).reshape(-1, 3).contiguous()
    keep += [pts, ids, noise]
    reg.num_background_points = pts.shape[0]
    reg.background_points = pts.data_ptr()
    reg.background_warp_ids = ids.data_ptr()
    reg.background_noise = None if noise is None else noise.data_ptr()
    reg.background_loss_weight = float(sp.background_loss_weight) if sp else 0.0
  return reg, keep


def value_and_grad(model, params, batch, warp_extra, rngs=None, chunk_rays=256, t_rand=None,
                   u_rand=None, grads=None, reg=None):
  """(loss dict, flat gradient) of the training loss (training.py:171-259, 263-264): the
  photometric terms and, with `reg` (make_reg), the regularisers.
  `grads` (flat, zeroed by the caller) may be passed to accumulate into."""
  dev = model.device
  origins = _prep_f32(batch['origins'], dev)
  directions = _prep_f32(batch['directions'], dev)
  B = origins.shape[0]
  viewdirs = _prep_f32(batch['viewdirs'], dev) if 'viewdirs' in batch else None
  md = batch.get('metadata', {})
  enc = model.warp_metadata_encoder_type if model.use_warp else None
  if enc == 'time':
    # models.py:252-254: the warp field reads metadata['time'] (B,1) float32
    t = md.get('time')
    warp_id = None if t is None else _prep_f32(t, dev).reshape(-1)
  else:
    warp_id = _prep_ids(md.get('warp'), dev) if model.use_warp else None
  if enc in ('time', 'blend') and warp_id is None:
    raise KeyError(f"batch['metadata']['{'time' if enc == 'time' else 'warp'}'] is required")
  app_id = _prep_ids(md.get('appearance'), dev) if model.use_appearance_metadata else None
  cam_id = _prep_ids(md.get('camera'), dev) if model.use_camera_metadata else None
  target = _prep_f32(batch['rgb'], dev)[..., :3].contiguous()
  if t_rand is None and u_rand is None:
    t_rand, u_rand = model._draws(rngs, B)
  t_rand = None if t_rand is None else _prep_f32(t_rand, dev)
  u_rand = None if u_rand is None else _prep_f32(u_rand, dev)
  hd = model.handle(B)
  hd.set_params(params)
  model._set_time_alpha(hd, (warp_extra or {}).get('time_alpha'))
  n = len(hd.param_specs)
  numels = [r * c for _, r, c in hd.param_specs]
  if grads is None:
    grads = torch.zeros(sum(numels), device=dev, dtype=torch.float32)
  ptrs, off = (ctypes.c_void_p * n)(), 0
  for i, k in enumerate(numels):
    ptrs[i] = grads.data_ptr() + 4 * off
    off += k
  loss = torch.zeros(16, device=dev)
  reg_struct, keep = reg if isinstance(reg, tuple) else (reg, None)
  with torch.cuda.device(dev):
    _lib.check(hd.lib.nfb_train_value_and_grad_reg(
        hd.h, B, _ptr(origins), _ptr(directions), _ptr(viewdirs), _ptr(warp_id), _ptr(app_id),
        _ptr(cam_id), float((warp_extra or {}).get('alpha', 0.0)), _ptr(t_rand), _ptr(u_rand), 0,
        _ptr(target), int(chunk_rays), ctypes.byref(reg_struct) if reg_struct is not None else None,
        ptrs, (ctypes.c_longlong * n)(*numels), n, _ptr(loss), _stream()))
  del keep
  out = {'coarse': loss[0], 'fine': loss[1]}
  if reg_struct is not None:
    out.update({'elastic': loss[2], 'elastic_residual': loss[3], 'jacobian_det': loss[4],
                'jacobian_div': loss[5], 'jacobian_curl': loss[6], 'warp_reg_coarse': loss[7],
                'warp_reg_residual_coarse': loss[8], 'warp_reg_fine': loss[9],
                'warp_reg_residual_fine': loss[10], 'background': loss[11]})
  return out, grads


def grads_to_tree(model, grads):
  """Flat gradient -> pytree with the Flax names (views)."""
  hd = model.handle(1)
  tree, off = {}, 0
  for name, rows, cols in hd.param_specs:
    t = tree
    parts = name.split('/')
    for part in parts[:-1]:
      t = t.setdefault(part, {})
    shape = (cols,) if parts[-1] == 'bias' else (rows, cols)
    t[parts[-1]] = grads[off:off + rows * cols].view(shape)
    off += rows * cols
  return tree


def train_step(model, rng_key, state, batch, scalar_params, use_elastic_loss=False,
               elastic_reduce_method='median', elastic_loss_type='log_svals',
               use_background_loss=False, use_warp_reg_loss=False, chunk_rays=256,
               timings=None):
  """One optimisation step (training.py:138-271).  Returns (new_state, stats, rng_key).

  timings (optional dict) receives 'value_and_grad_ms', 'all_reduce_ms', 'adam_ms' measured
  with CUDA events on the current stream."""
  reg = None
  if use_elastic_loss or use_warp_reg_loss or use_background_loss:
    bg = {}
    if use_background_loss:
      # training.py:122-126: ids ~ random.choice(key, model.warp_ids), noise ~ noise_std * N(0, 1);
      # integer ids for every encoder ('time' encodes float(id), as the reference does)
      pts = torch.as_tensor(batch['background_points']).reshape(-1, 3)
      gen = torch.Generator().manual_seed(int(rng_key) if not isinstance(rng_key, torch.Generator) else rng_key.seed())
      warp_ids = torch.as_tensor(list(model.warp_ids), dtype=torch.int64)
      bg['background_points'] = pts
      bg['background_warp_ids'] = batch.get(
          'background_warp_ids', warp_ids[torch.randint(len(warp_ids), (pts.shape[0],), generator=gen)])
      bg['background_noise'] = batch.get(
          'background_noise',
          scalar_params.background_noise_std * torch.randn(pts.shape[0], 3, generator=gen))
    reg = make_reg(model, scalar_params, use_elastic_loss, elastic_reduce_method, elastic_loss_type,
                   use_background_loss, use_warp_reg_loss, **bg)
  opt = state.optimizer
  ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timings is not None else None
  if ev:
    ev[0].record()
  params = opt.target['model']
  model.invalidate_params()     # the Adam kernel rewrote the flat vector under the views
  losses, grads = value_and_grad(model, params, batch, state.warp_extra,
                                 rngs={'coarse': rng_key, 'fine': rng_key}, chunk_rays=chunk_rays, reg=reg)
  if ev:
    ev[1].record()
  # stats of _compute_loss_and_stats (training.py:171-226)
  stats = {lv: {'loss/rgb': losses[lv], 'loss/total': losses[lv], 'metric/psnr': -10.0 * torch.log10(losses[lv])}
           for lv in ('coarse', 'fine') if lv in losses}
  if use_elastic_loss:
    c = stats['coarse']
    c['loss/elastic'] = losses['elastic']
    c['residual/elastic'] = losses['elastic_residual']
    c['loss/total'] = c['loss/total'] + scalar_params.elastic_loss_weight * losses['elastic']
    c['metric/jacobian_det'] = losses['jacobian_det']
    c['metric/jacobian_div'] = losses['jacobian_div']
    c['metric/jacobian_curl'] = losses['jacobian_curl']
  if use_warp_reg_loss:
    for lv in stats:
      stats[lv]['loss/warp_reg'] = losses['warp_reg_' + lv]
      stats[lv]['residual/warp_reg'] = losses['warp_reg_residual_' + lv]
      stats[lv]['loss/total'] = stats[lv]['loss/total'] + scalar_params.warp_reg_loss_weight * losses['warp_reg_' + lv]
  if use_background_loss:
    stats['background_loss'] = losses['background']
  if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
    # jax.lax.pmean(grad, 'batch') (training.py:266): one collective over the flat vector
    dist.all_reduce(grads)
    grads /= dist.get_world_size()
  if ev:
    ev[2].record()
  opt.apply_gradient(grads, learning_rate=scalar_params.learning_rate)
  if ev:
    ev[3].record()
    ev[3].synchronize()
    timings['value_and_grad_ms'] = ev[0].elapsed_time(ev[1])
    timings['all_reduce_ms'] = ev[1].elapsed_time(ev[2])
    timings['adam_ms'] = ev[2].elapsed_time(ev[3])
  return state, stats, rng_key
