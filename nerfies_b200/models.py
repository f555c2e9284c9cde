"""Host-side mirror of nerfies/models.py: NerfModel / construct_nerf.

The arithmetic runs in libnerfies_b200.so (hand-written sm_100a CUDA) through
the C ABI of include/nerfies_b200.h; this module keeps the reference's call
surface on top of it (SURVEY.md §8b):

  model, params = construct_nerf(key, config, batch_size, appearance_ids,
                                 camera_ids, warp_ids, near, far, ...)
  out = model.apply({'params': params}, rays_dict, warp_extra=...,
                    rngs={'coarse': k0, 'fine': k1}, mutable=False)
      -> {'coarse': {'rgb','depth','med_depth','acc'[,...]}, 'fine': {...}}

with torch CUDA tensors where the reference has jnp arrays.  Parameter pytrees
use the reference's Flax names, so a converted Flax checkpoint drops in.
"""
import ctypes
import math
from typing import Any, Dict, Mapping, Optional, Sequence

import torch

from nerfies_b200 import _lib
from nerfies_b200 import configs


def _mask(skips) -> int:
  m = 0
  for s in skips:
    m |= 1 << int(s)
  return m


def _ptr(t: Optional[torch.Tensor]):
  return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
  return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _prep_f32(t, device, shape_last=None):
  t = torch.as_tensor(t)
  t = t.to(device=device, dtype=torch.float32).contiguous()
  return t


def _prep_ids(t, device):
  """metadata ids arrive as (B,1) uint32 (models.py:469-473); the ABI wants (B)."""
  if t is None:
    return None
  t = torch.as_tensor(t)
  if t.dim() > 1:
    # (B,1) -> (B); an empty batch cannot be reshaped with -1.
    t = t.reshape(t.shape[0], -1)[:, 0] if t.numel() else t.reshape(0)
  # torch has no first-class uint32 arithmetic: carry the bits in int32.
  return t.to(device=device, dtype=torch.int32).contiguous()


class _Handle:
  """Owns one nfb_handle (one per model per device)."""

  def __init__(self, cfg: _lib.NfbConfig, max_rays: int, device):
    self.lib = _lib.load()
    self.device = device
    self.max_rays = max_rays
    h = ctypes.c_void_p()
    with torch.cuda.device(device):
      _lib.check(self.lib.nfb_create(ctypes.byref(cfg), max_rays,
                                     ctypes.byref(h)))
    self.h = h
    self.param_key = None
    n = self.lib.nfb_param_count(self.h)
    self.param_specs = []
    buf = ctypes.create_string_buffer(256)
    for i in range(n):
      r, c = ctypes.c_longlong(), ctypes.c_longlong()
      _lib.check(self.lib.nfb_param_info(self.h, i, buf, 256, ctypes.byref(r),
                                         ctypes.byref(c)))
      self.param_specs.append((buf.value.decode(), r.value, c.value))

  def close(self):
    if self.h is not None:
      self.lib.nfb_destroy(self.h)
      self.h = None

  def __del__(self):
    try:
      self.close()
    except Exception:  # pylint: disable=broad-except
      pass

  def set_params(self, params: Mapping[str, Any], partial: bool = False):
    """Uploads the parameter pytree.  partial=True (warp_field.apply with the warp
    subtree only): parameters missing from `params` keep the tensors of the last
    upload, or zeros when there was none."""
    tensors = []
    last = getattr(self, '_keepalive', None)
    for idx, (name, rows, cols) in enumerate(self.param_specs):
      node = params
      missing = False
      for part in name.split('/'):
        if not isinstance(node, Mapping) or part not in node:
          missing = True
          break
        node = node[part]
      if missing:
        if not partial or name.startswith('warp_field/'):
          raise KeyError(f'parameter {name!r} missing from the params pytree')
        tensors.append(last[idx] if last is not None else
                       torch.zeros(rows * cols, device=self.device))
        continue
      t = node
      if not torch.is_tensor(t):
        t = torch.as_tensor(t)
      if t.numel() != rows * cols:
        raise ValueError(f'parameter {name}: shape {tuple(t.shape)} does not '
                         f'hold {rows}x{cols} elements')
      tensors.append(t.to(device=self.device, dtype=torch.float32).contiguous())
    key = tuple((t.data_ptr(), t._version) for t in tensors)
    if key == self.param_key:
      return
    n = len(tensors)
    ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in tensors])
    numels = (ctypes.c_longlong * n)(*[t.numel() for t in tensors])
    _lib.check(self.lib.nfb_set_params(self.h, ptrs, numels, n, _stream()))
    self.param_key = key
    self._keepalive = tensors  # until the stream has consumed them


class NerfModel:
  """Mirror of nerfies.models.NerfModel (models.py:31-375), forward only."""

  def __init__(self, *, num_coarse_samples, num_fine_samples, use_viewdirs,
               near, far, noise_std, nerf_trunk_depth, nerf_trunk_width,
               nerf_rgb_branch_depth, nerf_rgb_branch_width, nerf_skips,
               alpha_channels, rgb_channels, use_stratified_sampling,
               num_nerf_point_freqs, num_nerf_viewdir_freqs, appearance_ids,
               camera_ids, warp_ids, num_appearance_features,
               num_camera_features, num_warp_features, num_warp_freqs,
               activation='relu', sigma_activation='relu',
               use_white_background=False, use_linear_disparity=False,
               use_sample_at_infinity=True, warp_field_type='se3',
               warp_metadata_encoder_type='glo', use_appearance_metadata=False,
               use_camera_metadata=False, use_warp=False,
               use_warp_jacobian=False, use_weights=False,
               use_trunk_condition=False, use_alpha_condition=False,
               use_rgb_condition=False, warp_kwargs=None, precision='fp32',
               batch_size=8192, device=None):
    self.num_coarse_samples = int(num_coarse_samples)
    self.num_fine_samples = int(num_fine_samples)
    self.use_viewdirs = bool(use_viewdirs)
    self.near = float(near)
    self.far = float(far)
    self.noise_std = noise_std
    self.nerf_trunk_depth = int(nerf_trunk_depth)
    self.nerf_trunk_width = int(nerf_trunk_width)
    self.nerf_rgb_branch_depth = int(nerf_rgb_branch_depth)
    self.nerf_rgb_branch_width = int(nerf_rgb_branch_width)
    self.nerf_skips = tuple(nerf_skips)
    self.alpha_channels = int(alpha_channels)
    self.rgb_channels = int(rgb_channels)
    self.use_stratified_sampling = bool(use_stratified_sampling)
    self.num_nerf_point_freqs = int(num_nerf_point_freqs)
    self.num_nerf_viewdir_freqs = int(num_nerf_viewdir_freqs)
    self.appearance_ids = list(appearance_ids)
    self.camera_ids = list(camera_ids)
    self.warp_ids = list(warp_ids)
    self.num_appearance_features = int(num_appearance_features)
    self.num_camera_features = int(num_camera_features)
    self.num_warp_features = int(num_warp_features)
    self.num_warp_freqs = int(num_warp_freqs)
    self.activation = configs.activation_name(activation)
    self.sigma_activation = configs.activation_name(sigma_activation)
    self.use_white_background = bool(use_white_background)
    self.use_linear_disparity = bool(use_linear_disparity)
    self.use_sample_at_infinity = bool(use_sample_at_infinity)
    self.warp_field_type = warp_field_type
    self.warp_metadata_encoder_type = warp_metadata_encoder_type
    self.use_appearance_metadata = bool(use_appearance_metadata)
    self.use_camera_metadata = bool(use_camera_metadata)
    self.use_warp = bool(use_warp)
    self.use_warp_jacobian = bool(use_warp_jacobian)
    self.use_weights = bool(use_weights)
    self.use_trunk_condition = bool(use_trunk_condition)
    self.use_alpha_condition = bool(use_alpha_condition)
    self.use_rgb_condition = bool(use_rgb_condition)
    self.warp_kwargs = dict(warp_kwargs or {})
    self.precision = precision
    self.batch_size = int(batch_size)
    if device is None:
      # parameters may be built without a GPU (host-logic tests); apply() needs one.
      device = 'cuda' if torch.cuda.is_available() else 'cpu'
    self.device = torch.device(device)
    if self.device.type == 'cuda' and self.device.index is None:
      self.device = torch.device('cuda', torch.cuda.current_device())
    self._handle = None

    if noise_std is not None and noise_std > 0.0 and use_stratified_sampling:
      # The reference itself cannot run this branch: NerfModel.render_samples hands the
      # NerfMLP's output DICT to noise_regularize, which indexes it as an array
      # (models.py:272-275 vs model_utils.py:278-280) -> TypeError.  Same error type here.
      raise TypeError("noise_std > 0 with stratified sampling: the reference's "
                      "noise_regularize (model_utils.py:266-282) raises on the NerfMLP's dict "
                      'output (models.py:274); there is no behaviour to reproduce')
    if self.use_warp:
      if warp_field_type not in ('se3', 'translation'):
        raise ValueError(f'Unknown warp field type: {warp_field_type!r}')
      ok_enc = ('glo', 'time') if warp_field_type == 'se3' else ('glo', 'time', 'blend')
      if warp_metadata_encoder_type not in ok_enc:
        # warping.py:121-123 / 258-260
        raise ValueError(f'Unknown metadata encoder type {warp_metadata_encoder_type}')
      allowed = ({'trunk_depth', 'trunk_width', 'skips', 'use_pivot', 'use_translation',
                  'metadata_encoder_num_freqs'} if warp_field_type == 'se3' else
                 {'depth', 'hidden_channels', 'skips', 'metadata_encoder_num_freqs'})
      extra = set(self.warp_kwargs) - allowed
      if extra:
        raise NotImplementedError(
            f'warp_kwargs {sorted(extra)} not supported (rotation/pivot/translation branch '
            'depths > 0, min/max_freq_log2, use_identity_map=False, custom initialisers)')
    if precision not in _lib.PRECISIONS:
      raise ValueError(f'precision must be one of {list(_lib.PRECISIONS)}')

  # Same derived attributes as the reference (models.py:121-131).
  @property
  def num_appearance_embeddings(self):
    return max(self.appearance_ids) + 1

  @property
  def num_warp_embeddings(self):
    return max(self.warp_ids) + 1

  @property
  def num_camera_embeddings(self):
    return max(self.camera_ids) + 1

  @property
  def warp_trunk_depth(self):
    k = 'trunk_depth' if self.warp_field_type == 'se3' else 'depth'
    return int(self.warp_kwargs.get(k, 6))

  @property
  def warp_trunk_width(self):
    k = 'trunk_width' if self.warp_field_type == 'se3' else 'hidden_channels'
    return int(self.warp_kwargs.get(k, 128))

  @property
  def warp_skips(self):
    return tuple(self.warp_kwargs.get('skips', (4,)))

  @property
  def metadata_encoder_num_freqs(self):
    return int(self.warp_kwargs.get('metadata_encoder_num_freqs', 1))

  @property
  def warp_use_pivot(self):
    return bool(self.warp_kwargs.get('use_pivot', False))

  @property
  def warp_use_translation(self):
    return bool(self.warp_kwargs.get('use_translation', False))

  # -- C ABI plumbing ---------------------------------------------------------
  def nfb_config(self) -> _lib.NfbConfig:
    c = _lib.NfbConfig()
    c.num_coarse_samples = self.num_coarse_samples
    c.num_fine_samples = self.num_fine_samples
    c.num_nerf_point_freqs = self.num_nerf_point_freqs
    c.num_nerf_viewdir_freqs = self.num_nerf_viewdir_freqs
    c.num_warp_freqs = self.num_warp_freqs
    c.nerf_trunk_depth = self.nerf_trunk_depth
    c.nerf_trunk_width = self.nerf_trunk_width
    c.nerf_rgb_branch_depth = self.nerf_rgb_branch_depth
    c.nerf_rgb_branch_width = self.nerf_rgb_branch_width
    c.nerf_skips_mask = _mask(self.nerf_skips)
    c.alpha_channels = self.alpha_channels
    c.rgb_channels = self.rgb_channels
    c.warp_field_type = (_lib.WARP_TYPES[self.warp_field_type]
                         if self.use_warp else 0)
    c.warp_trunk_depth = self.warp_trunk_depth
    c.warp_trunk_width = self.warp_trunk_width
    c.warp_skips_mask = _mask(self.warp_skips)
    c.num_warp_features = self.num_warp_features
    c.num_appearance_features = self.num_appearance_features
    c.num_camera_features = self.num_camera_features
    c.num_warp_embeddings = self.num_warp_embeddings
    c.num_appearance_embeddings = self.num_appearance_embeddings
    c.num_camera_embeddings = self.num_camera_embeddings
    c.use_viewdirs = int(self.use_viewdirs)
    c.use_appearance_metadata = int(self.use_appearance_metadata)
    c.use_camera_metadata = int(self.use_camera_metadata)
    c.use_trunk_condition = int(self.use_trunk_condition)
    c.use_alpha_condition = int(self.use_alpha_condition)
    c.use_rgb_condition = int(self.use_rgb_condition)
    c.activation = _lib.ACTIVATIONS[self.activation]
    c.sigma_activation = _lib.ACTIVATIONS[self.sigma_activation]
    c.use_white_background = int(self.use_white_background)
    c.use_linear_disparity = int(self.use_linear_disparity)
    c.use_sample_at_infinity = int(self.use_sample_at_infinity)
    c.near_plane = self.near
    c.far_plane = self.far
    c.precision = _lib.PRECISIONS[self.precision]
    c.warp_metadata_encoder = _lib.WARP_ENCODERS[self.warp_metadata_encoder_type]
    c.time_encoder_num_freqs = self.metadata_encoder_num_freqs
    c.warp_use_pivot = int(self.warp_use_pivot)
    c.warp_use_translation = int(self.warp_use_translation)
    return c

  def handle(self, num_rays: int = 0) -> _Handle:
    if not torch.cuda.is_available():
      raise RuntimeError('nerfies_b200 needs a CUDA device (sm_100a); there is '
                         'no CPU fallback')
    want = max(self.batch_size, num_rays)
    if self._handle is None or self._handle.max_rays < want:
      if self._handle is not None:
        self._handle.close()
      self._handle = _Handle(self.nfb_config(), want, self.device)
    return self._handle

  def invalidate_params(self):
    """Forces the next call to re-upload the parameters (their storage was rewritten in place
    by a kernel torch does not see, e.g. nfb_adam_step)."""
    if self._handle is not None:
      self._handle.param_key = None

  def kernel_launches(self) -> int:
    if self._handle is None:
      return 0
    return int(self._handle.lib.nfb_kernel_launches(self._handle.h))

  @staticmethod
  def create_warp_field(model, num_batch_dims):
    """models.py:133-142: a warp field sharing the model's configuration."""
    del num_batch_dims  # points are always flattened to (P, 3) here.
    return WarpField(model)

  def _draws(self, rngs, num_rays):
    """Uniform draws of the stratified path (model_utils.py:65,162).  The
    reference folds jax.random threefry keys; these are torch Philox draws
    seeded from the given keys - same distribution, not the same bits."""
    if not self.use_stratified_sampling:
      return None, None

    def gen(key, salt):
      g = torch.Generator(device=self.device)
      seed = 0
      if key is not None:
        k = torch.as_tensor(key).flatten().tolist() if not isinstance(
            key, int) else [key]
        for v in k:
          seed = (seed * 1000003 + int(v)) % (2**62)
      g.manual_seed(seed + salt)
      return g

    rngs = rngs or {}
    t = torch.rand(num_rays, self.num_coarse_samples, device=self.device,
                   generator=gen(rngs.get('coarse'), 1))
    u = None
    if self.num_fine_samples > 0:
      u = torch.rand(num_rays, self.num_fine_samples, device=self.device,
                     generator=gen(rngs.get('fine'), 2))
    return t, u

  # -- forward ----------------------------------------------------------------
  def apply(self, variables, rays_dict, warp_extra=None, metadata_encoded=False,
            use_warp=True, return_points=False, return_weights=False,
            return_warp_jacobian=False, deterministic=False, rngs=None,
            mutable=False, t_rand=None, u_rand=None, _packed=False):
    """model.apply({'params': params}, rays_dict, warp_extra=..., rngs=...)
    as called at training.py:229-237 and eval.py:331-338 (models.py:289-375).

    Extra keyword arguments `t_rand` (B,Nc) / `u_rand` (B,Nf) inject the
    uniform draws of the stratified path (used by the parity tests).
    """
    del deterministic, mutable  # unused by the reference's __call__ as well.
    # models.py:345, 367: the coarse level returns Jacobians when either the call or the
    # model asks for them, the fine level only when the call does.
    jac_levels = []
    if use_warp and self.use_warp:
      if return_warp_jacobian or self.use_warp_jacobian:
        jac_levels.append('coarse')
      if return_warp_jacobian:
        jac_levels.append('fine')
    if jac_levels and metadata_encoded:
      raise NotImplementedError('warp Jacobians of metadata_encoded=True calls')
    want_points = return_points
    return_points = return_points or bool(jac_levels)       # the Jacobian is taken at the sample points
    params = variables['params']
    warp_extra = warp_extra or {'alpha': 0.0, 'time_alpha': 0.0}
    alpha = float(warp_extra.get('alpha', 0.0))
    time_alpha = warp_extra.get('time_alpha')
    dev = self.device
    origins = _prep_f32(rays_dict['origins'], dev)
    directions = _prep_f32(rays_dict['directions'], dev)
    if origins.dim() != 2 or origins.shape[-1] != 3:
      raise ValueError('origins must be (B, 3)')
    B = origins.shape[0]
    viewdirs = (_prep_f32(rays_dict['viewdirs'], dev)
                if 'viewdirs' in rays_dict else None)
    md = rays_dict.get('metadata', {})
    use_warp = self.use_warp and use_warp
    if metadata_encoded:
      # models.py:198-213,251 / warping.py:186-187: the metadata leaves are the
      # per-ray embeddings themselves, (B, num_*_features) float32.
      def enc(key, width, used):
        if not used:
          return None
        v = md.get(key)
        if v is None:
          return None
        v = _prep_f32(v, dev)
        if v.shape != (B, width):
          raise ValueError(f"metadata_encoded=True: metadata['{key}'] must be ({B}, {width}), "
                           f'got {tuple(v.shape)}')
        return v
      warp_id = enc('warp', self.num_warp_features, self.use_warp)
      app_id = enc('appearance', self.num_appearance_features, self.use_appearance_metadata)
      cam_id = enc('camera', self.num_camera_features, self.use_camera_metadata)
    else:
      if self.use_warp and self.warp_metadata_encoder_type == 'time':
        # models.py:252-254: the warp field reads metadata['time'] (B,1) float32
        t = md.get('time')
        warp_id = None if t is None else _prep_f32(t, dev).reshape(-1)
      else:
        warp_id = _prep_ids(md.get('warp'), dev) if self.use_warp else None
      app_id = (_prep_ids(md.get('appearance'), dev)
                if self.use_appearance_metadata else None)
      cam_id = (_prep_ids(md.get('camera'), dev)
                if self.use_camera_metadata else None)
    if self.use_warp and use_warp and warp_id is None:
      key = 'time' if self.warp_metadata_encoder_type == 'time' else 'warp'
      raise KeyError(f"rays_dict['metadata']['{key}'] is required")
    return_weights = self.use_weights or return_weights
    if t_rand is None and u_rand is None:
      t_rand, u_rand = self._draws(rngs, B)
    if t_rand is not None:
      t_rand = _prep_f32(t_rand, dev)
    if u_rand is not None:
      u_rand = _prep_f32(u_rand, dev)

    hd = self.handle(B)
    hd.set_params(params)
    lib, h = hd.lib, hd.h
    self._set_time_alpha(hd, time_alpha)
    nc, nf = self.num_coarse_samples, self.num_fine_samples
    flags = 0 if use_warp else _lib.FLAG_NO_WARP
    if metadata_encoded:
      flags |= _lib.FLAG_METADATA_ENCODED
    out = {}
    with torch.cuda.device(dev):
      out_c = torch.empty(B, 6, device=dev)
      w_c = torch.empty(B, nc, device=dev)
      out_f = torch.empty(B, 6, device=dev) if nf > 0 else None
      w_f = (torch.empty(B, nc + nf, device=dev)
             if nf > 0 and return_weights else None)
      if not return_points:
        _lib.check(lib.nfb_render_forward(
            h, B, _ptr(origins), _ptr(directions), _ptr(viewdirs),
            _ptr(warp_id), _ptr(app_id), _ptr(cam_id), alpha, _ptr(t_rand),
            _ptr(u_rand), flags, _ptr(out_c), _ptr(out_f), _ptr(w_c),
            _ptr(w_f), None, _stream()))
        pts = {}
      else:
        # staged path: exposes z_vals / warped points of both levels.
        pts = {}
        z_c = torch.empty(B, nc, device=dev)
        _lib.check(lib.nfb_coarse_z_vals(h, B, _ptr(t_rand), _ptr(z_c),
                                         _stream()))
        wp_c = torch.empty(B, nc, 3, device=dev)
        _lib.check(lib.nfb_render_samples(
            h, 0, B, nc, _ptr(z_c), _ptr(origins), _ptr(directions),
            _ptr(viewdirs), _ptr(warp_id), _ptr(app_id), _ptr(cam_id), alpha,
            flags, _ptr(out_c), _ptr(w_c), None, _ptr(wp_c), _stream()))
        pts['coarse'] = (z_c, wp_c)
        if nf > 0:
          z_f = torch.empty(B, nc + nf, device=dev)
          _lib.check(lib.nfb_sample_pdf(h, B, _ptr(z_c), _ptr(w_c),
                                        _ptr(u_rand), _ptr(z_f), _stream()))
          wp_f = torch.empty(B, nc + nf, 3, device=dev)
          _lib.check(lib.nfb_render_samples(
              h, 1, B, nc + nf, _ptr(z_f), _ptr(origins), _ptr(directions),
              _ptr(viewdirs), _ptr(warp_id), _ptr(app_id), _ptr(cam_id), alpha,
              flags, _ptr(out_f), _ptr(w_f), None, _ptr(wp_f), _stream()))
          pts['fine'] = (z_f, wp_f)

    def pack(o, w, level):
      ret = {'rgb': o[:, 0:3], 'depth': o[:, 3], 'med_depth': o[:, 4],
             'acc': o[:, 5]}
      if return_weights and w is not None:
        ret['weights'] = w
      if level in pts:
        z, wp = pts[level]
        points = origins[:, None, :] + z[:, :, None] * directions[:, None, :]
        if level in jac_levels:
          # jax.jacfwd(self.warp)(points, ...) for every sample (warping.py:385-387, models.py:265-266)
          S = z.shape[1]
          flat = points.reshape(-1, 3).contiguous()
          ids = warp_id[:, None].expand(B, S).reshape(-1).contiguous()
          jac = torch.empty(B * S, 3, 3, device=dev)
          with torch.cuda.device(dev):
            _lib.check(lib.nfb_warp_jacobian(h, B * S, _ptr(flat), _ptr(ids), alpha, None, _ptr(jac),
                                             _stream()))
          ret['warp_jacobian'] = jac.reshape(B, S, 3, 3)
        if want_points:
          ret['points'] = points
          if use_warp:
            ret['warped_points'] = wp
          ret['z_vals'] = z
      return ret

    if _packed:
      # evaluation.py: the (B,6) buffers the C ABI wrote (rgb3, depth, med_depth, acc) -
      # one contiguous block per level, so a frame's collective moves them unsplit
      return {'coarse': out_c, 'fine': out_f} if nf > 0 else {'coarse': out_c}
    out['coarse'] = pack(out_c, w_c, 'coarse')
    if nf > 0:
      out['fine'] = pack(out_f, w_f, 'fine')
    return out

  __call__ = apply

  def _set_time_alpha(self, hd, time_alpha):
    """warp_extra['time_alpha'] for the 'time' / 'blend' encoders (None -> the
    TimeEncoder's num_freqs, modules.py:318-319; 'blend' needs a number)."""
    if not self.use_warp or self.warp_metadata_encoder_type == 'glo':
      return
    if time_alpha is None:
      if self.warp_metadata_encoder_type == 'blend':
        raise TypeError("warp_extra['time_alpha'] is required by the 'blend' encoder (warping.py:132)")
      time_alpha = float(self.metadata_encoder_num_freqs)
    _lib.check(hd.lib.nfb_set_time_alpha(hd.h, float(time_alpha)))

  def apply_host(self, variables, rays_dict, warp_extra=None):
    """End-to-end call on HOST (numpy / CPU torch) buffers: pinned staging,
    H2D, render, D2H inside nfb_render_forward_host.  Deterministic path."""
    import numpy as np
    params = variables['params']
    alpha = float((warp_extra or {}).get('alpha', 0.0))
    f32 = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float32))
    origins, directions = f32(rays_dict['origins']), f32(rays_dict['directions'])
    B = origins.shape[0]
    viewdirs = f32(rays_dict['viewdirs']) if 'viewdirs' in rays_dict else None
    md = rays_dict.get('metadata', {})

    def ids(key, used):
      if not used or key not in md:
        return None
      a = np.asarray(md[key]).reshape(B, -1)[:, 0]
      return np.ascontiguousarray(a.astype(np.uint32))

    warp_id = ids('warp', self.use_warp)
    app_id = ids('appearance', self.use_appearance_metadata)
    cam_id = ids('camera', self.use_camera_metadata)
    hd = self.handle(B)
    hd.set_params(params)
    out_c = np.empty((B, 6), np.float32)
    out_f = np.empty((B, 6), np.float32)
    p = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    with torch.cuda.device(self.device):
      _lib.check(hd.lib.nfb_render_forward_host(
          hd.h, B, p(origins), p(directions), p(viewdirs), p(warp_id),
          p(app_id), p(cam_id), alpha, 0, p(out_c), p(out_f), _stream()))
    unpack = lambda o: {'rgb': o[:, 0:3], 'depth': o[:, 3],
                        'med_depth': o[:, 4], 'acc': o[:, 5]}
    out = {'coarse': unpack(out_c)}
    if self.num_fine_samples > 0:
      out['fine'] = unpack(out_f)
    return out


class WarpField:
  """warp_field.apply on free points (warping.py:355-389; training.py:122-131)."""

  def __init__(self, model: NerfModel):
    self.model = model

  def apply(self, variables, points, metadata, extra, return_jacobian=False,
            metadata_encoded=False):
    """`variables` = {'params': params['warp_field']} as the reference call site passes
    it (training.py:127-131) - or the whole model tree.  The given warp parameters
    are uploaded on every call whose tensors changed; with the subtree only, the
    non-warp parameters keep their last uploaded values (zeros if none were ever
    uploaded - the warp-only launch does not read them)."""
    m = self.model
    if return_jacobian and metadata_encoded:
      raise NotImplementedError('warp Jacobian of a metadata_encoded=True call')
    dev = m.device
    pts = _prep_f32(points, dev)
    shape = pts.shape
    pts = pts.reshape(-1, 3)
    P = pts.shape[0]
    if metadata_encoded:                                   # warping.py:186-187, 378
      ids = _prep_f32(metadata, dev).reshape(P, -1)
      if ids.shape[1] != m.num_warp_features:
        raise ValueError(f'metadata_encoded=True: metadata must be (P, {m.num_warp_features})')
      ids = ids.contiguous()
      flags = _lib.FLAG_METADATA_ENCODED
    elif m.warp_metadata_encoder_type == 'time':
      ids, flags = _prep_f32(metadata, dev).reshape(-1), 0
    else:
      ids, flags = _prep_ids(torch.as_tensor(metadata).reshape(P, -1), dev), 0
    hd = m.handle(P)
    p = variables['params']
    hd.set_params(p if 'warp_field' in p else {'warp_field': p}, partial=True)
    m._set_time_alpha(hd, extra.get('time_alpha'))
    out = torch.empty_like(pts)
    with torch.cuda.device(dev):
      _lib.check(hd.lib.nfb_warp_forward(
          hd.h, P, _ptr(pts), _ptr(ids), float(extra.get('alpha', 0.0)), flags,
          _ptr(out), _stream()))
      ret = {'warped_points': out.reshape(shape)}
      if return_jacobian:                                  # warping.py:385-387
        jac = torch.empty(P, 3, 3, device=dev)
        _lib.check(hd.lib.nfb_warp_jacobian(hd.h, P, _ptr(pts), _ptr(ids), float(extra.get('alpha', 0.0)),
                                            None, _ptr(jac), _stream()))
        ret['jacobian'] = jac.reshape(*shape[:-1], 3, 3)
    return ret


# ---------------------------------------------------------------------------
# construct_nerf (models.py:378-489)
# ---------------------------------------------------------------------------
def _generator(key, device):
  g = torch.Generator(device='cpu')
  if isinstance(key, torch.Generator):
    return key
  seed = 0
  for v in torch.as_tensor(key).flatten().tolist():
    seed = (seed * 1000003 + int(v)) % (2**62)
  g.manual_seed(seed)
  return g


def init_params(model: NerfModel, key) -> Dict[str, Any]:
  """Random parameters with the reference's initialisers (SURVEY §8a R12):
  glorot/xavier-uniform Dense kernels (modules.py:107-108,127-139;
  warping.py:237), zero biases, warp heads U[0,1e-4) (warping.py:238-240),
  embeddings U[0,0.05) (glo.py:33).  Pytree keys are the Flax names."""
  g = _generator(key, model.device)
  dev = model.device

  def glorot(fi, fo):
    a = math.sqrt(6.0 / (fi + fo))
    return ((torch.rand(fi, fo, generator=g) * 2 - 1) * a).to(dev)

  def dense(fi, fo, scale=None):
    k = glorot(fi, fo) if scale is None else (
        torch.rand(fi, fo, generator=g) * scale).to(dev)
    return {'kernel': k, 'bias': torch.zeros(fo, device=dev)}

  def mlp(in_dim, depth, width, skips, out=0, out_scale=None):
    p, d = {}, in_dim
    for i in range(depth):
      if i in skips:
        d += in_dim
      p[f'hidden_{i}'] = dense(d, width)
      d = width
    if out:
      p['logit'] = dense(d, out, out_scale)
    return p

  def embed(n, f):
    return {'embed': {'embedding': (torch.rand(n, f, generator=g) * 0.05).to(dev)}}

  params = {}
  if model.use_warp:
    dw = 3 + 6 * model.num_warp_freqs + model.num_warp_features
    glo = lambda: embed(model.num_warp_embeddings, model.num_warp_features)
    # modules.TimeEncoder (modules.py:297-315): xavier hidden layers, U[0,0.05) output layer
    tenc = lambda: {'mlp': mlp(1 + 2 * model.metadata_encoder_num_freqs, 6, 64, (4,),
                               model.num_warp_features, 0.05)}
    enc = model.warp_metadata_encoder_type
    if enc == 'glo':
      wf = {'metadata_encoder': glo()}
    elif enc == 'time':
      wf = {'metadata_encoder': tenc()}
    else:
      wf = {'glo_encoder': glo(), 'time_encoder': tenc()}
    if model.warp_field_type == 'se3':
      wf['trunk'] = mlp(dw, model.warp_trunk_depth, model.warp_trunk_width,
                        model.warp_skips)
      wf['branches_w'] = {'logit': dense(model.warp_trunk_width, 3, 1e-4)}
      wf['branches_v'] = {'logit': dense(model.warp_trunk_width, 3, 1e-4)}
      if model.warp_use_pivot:
        wf['branches_p'] = {'logit': dense(model.warp_trunk_width, 3, 1e-4)}
      if model.warp_use_translation:
        wf['branches_t'] = {'logit': dense(model.warp_trunk_width, 3, 1e-4)}
    else:
      wf['mlp'] = mlp(dw, model.warp_trunk_depth, model.warp_trunk_width,
                      model.warp_skips, 3, 1e-4)
    params['warp_field'] = wf
  if model.use_appearance_metadata:
    params['appearance_encoder'] = embed(model.num_appearance_embeddings,
                                         model.num_appearance_features)
  if model.use_camera_metadata:
    params['camera_encoder'] = embed(model.num_camera_embeddings,
                                     model.num_camera_features)
  a = model.num_appearance_features
  tc = a if (model.use_appearance_metadata and model.use_trunk_condition) else 0
  ac = a if (model.use_appearance_metadata and model.use_alpha_condition) else 0
  rc = ac + (3 + 6 * model.num_nerf_viewdir_freqs if model.use_viewdirs else 0)
  if model.use_camera_metadata:
    rc += model.num_camera_features
  dp = 3 + 6 * model.num_nerf_point_freqs
  w = model.nerf_trunk_width
  for level in ['coarse'] + (['fine'] if model.num_fine_samples > 0 else []):
    m = {'MLP_0': mlp(dp + tc, model.nerf_trunk_depth, w, model.nerf_skips)}
    if ac or rc:
      m['bottleneck'] = dense(w, w)
    m['MLP_1'] = mlp(w + rc, model.nerf_rgb_branch_depth,
                     model.nerf_rgb_branch_width, (), model.rgb_channels)
    m['MLP_2'] = mlp(w + ac, 0, 128, (), model.alpha_channels)
    params[f'nerf_mlps_{level}'] = m
  return params


def construct_nerf(key, config: configs.ModelConfig, batch_size: int,
                   appearance_ids: Sequence[int], camera_ids: Sequence[int],
                   warp_ids: Sequence[int], near: float, far: float,
                   use_warp_jacobian: bool = False, use_weights: bool = False,
                   precision: str = 'fp32', device=None):
  """Same signature and return value as models.construct_nerf
  (models.py:378-489) plus the B200-only keywords `precision` and `device`.

  Note: like the reference, `use_trunk_condition` is NOT forwarded from the
  config (models.py:424-463)."""
  model = NerfModel(
      num_coarse_samples=config.num_coarse_samples,
      num_fine_samples=config.num_fine_samples,
      use_viewdirs=config.use_viewdirs, near=near, far=far,
      noise_std=config.noise_std, nerf_trunk_depth=config.nerf_trunk_depth,
      nerf_trunk_width=config.nerf_trunk_width,
      nerf_rgb_branch_depth=config.nerf_rgb_branch_depth,
      nerf_rgb_branch_width=config.nerf_rgb_branch_width,
      use_alpha_condition=config.use_alpha_condition,
      use_rgb_condition=config.use_rgb_condition, activation=config.activation,
      sigma_activation=config.sigma_activation, nerf_skips=config.nerf_skips,
      alpha_channels=config.alpha_channels, rgb_channels=config.rgb_channels,
      use_stratified_sampling=config.use_stratified_sampling,
      use_white_background=config.use_white_background,
      use_sample_at_infinity=config.use_sample_at_infinity,
      num_nerf_point_freqs=config.num_nerf_point_freqs,
      num_nerf_viewdir_freqs=config.num_nerf_viewdir_freqs,
      use_linear_disparity=config.use_linear_disparity,
      use_warp_jacobian=use_warp_jacobian, use_weights=use_weights,
      use_appearance_metadata=config.use_appearance_metadata,
      use_camera_metadata=config.use_camera_metadata, use_warp=config.use_warp,
      appearance_ids=appearance_ids, camera_ids=camera_ids, warp_ids=warp_ids,
      num_appearance_features=config.appearance_metadata_dims,
      num_camera_features=config.camera_metadata_dims,
      num_warp_freqs=config.num_warp_freqs,
      num_warp_features=config.num_warp_features,
      warp_field_type=config.warp_field_type,
      warp_metadata_encoder_type=config.warp_metadata_encoder_type,
      warp_kwargs=dict(config.warp_kwargs), precision=precision,
      batch_size=batch_size, device=device)
  params = init_params(model, key)
  return model, params
