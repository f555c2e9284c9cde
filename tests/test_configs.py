"""ModelConfig surface + the gin subset (nerfies/configs.py, configs/*.gin)."""
import dataclasses
import os

import pytest

from nerfies_b200 import configs

GIN = '''
# macros, lazily resolved (a later assignment wins, like gin)
num_warp_freqs = 8
SCHED = {
  'type': 'linear',
  'initial_value': 0.0,
  'final_value': %num_warp_freqs,   # trailing comment
  'num_steps': 80000,
}
batch_size = 6144
ModelConfig.sigma_activation = @nn.softplus
ModelConfig.use_warp = True
ModelConfig.warp_field_type = 'se3'
ModelConfig.num_warp_freqs = %num_warp_freqs
ModelConfig.num_coarse_samples = 128
TrainConfig.batch_size = %batch_size
TrainConfig.warp_alpha_schedule = %SCHED
TrainConfig.elastic_loss_weight_schedule = {
  'type': 'piecewise',
  'schedules': [
    (50000, ('constant', 0.01)),
    (100000, ('cosine_easing', 0.01, 1e-8, 100000)),
  ]
}
EvalConfig.chunk = 4096
SomethingElse.value = 3
num_warp_freqs = 6
'''


@pytest.fixture(autouse=True)
def _clear():
  configs.clear_config()
  yield
  configs.clear_config()


def test_defaults_match_reference():
  # nerfies/configs.py:37-105.
  c = configs.ModelConfig()
  assert (c.num_coarse_samples, c.num_fine_samples) == (64, 128)
  assert (c.nerf_trunk_depth, c.nerf_trunk_width) == (8, 256)
  assert (c.nerf_rgb_branch_depth, c.nerf_rgb_branch_width) == (1, 128)
  assert c.nerf_skips == (4,) and c.num_nerf_point_freqs == 10
  assert c.num_nerf_viewdir_freqs == 4 and c.use_stratified_sampling
  assert c.warp_field_type == 'translation' and not c.use_warp
  assert c.activation == 'relu' and c.sigma_activation == 'relu'
  assert configs.EvalConfig().chunk == 8192
  with pytest.raises(ValueError):
    configs.TrainConfig()   # batch_size = gin.REQUIRED


def test_gin_subset():
  configs.parse_config(GIN)
  m = configs.ModelConfig(use_stratified_sampling=False)
  assert m.sigma_activation == 'softplus' and m.use_warp
  assert m.num_warp_freqs == 6            # lazy macro resolution
  assert m.num_coarse_samples == 128 and not m.use_stratified_sampling
  t = configs.TrainConfig()
  assert t.batch_size == 6144
  assert t.warp_alpha_schedule['final_value'] == 6
  assert t.elastic_loss_weight_schedule['schedules'][1][1][0] == 'cosine_easing'
  assert configs.EvalConfig().chunk == 4096


def test_gin_files_and_includes(tmp_path):
  (tmp_path / 'base.gin').write_text(
      "ModelConfig.num_fine_samples = 32\nfar = 2.5\n")
  (tmp_path / 'top.gin').write_text(
      "include 'base.gin'\nModelConfig.num_coarse_samples = 16\n")
  configs.parse_config_files_and_bindings(
      [str(tmp_path / 'top.gin')], ['ModelConfig.nerf_trunk_width = 64'])
  m = configs.ModelConfig()
  assert (m.num_coarse_samples, m.num_fine_samples, m.nerf_trunk_width) == (
      16, 32, 64)


def test_reference_gin_files_if_present():
  # Verbatim copies of the reference's configs/*.gin (Apache-2.0), including the
  # files they include.
  root = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'configs')
  expected = {'gpu_quarterhd.gin': (6144, 128, 128, 8, 8),
              'gpu_fullhd.gin': (4096, 256, 256, 10, 8),
              'gpu_vrig_paper.gin': (6144, 128, 128, 8, 6),
              'test_local.gin': (1024, 64, 64, 10, 8)}
  for f, (bs, nc, nf, fp, fw) in expected.items():
    configs.clear_config()
    configs.parse_config_files_and_bindings([os.path.join(root, f)])
    m, t = configs.ModelConfig(), configs.TrainConfig()
    assert (t.batch_size, m.num_coarse_samples, m.num_fine_samples,
            m.num_nerf_point_freqs, m.num_warp_freqs) == (bs, nc, nf, fp, fw)
    assert m.sigma_activation == 'softplus' and m.warp_field_type == 'se3'


def test_activation_names():
  assert configs.activation_name('softplus') == 'softplus'

  def relu(x):
    return x
  assert configs.activation_name(relu) == 'relu'
  with pytest.raises(ValueError):
    configs.activation_name('gelu')
  assert dataclasses.is_dataclass(configs.ModelConfig)
