"""Pin the oracle (oracle/*.py) against fixtures produced by the real reference
(tools/make_golden.py).  CPU only; these are the `-m "not gpu"` parity anchors."""
import numpy as np
import pytest
import torch

from helpers import golden, golden_config, seeded_model, rel_l2
from oracle import ncsnpp_oracle as NO
from oracle import sampling_oracle as SO


@pytest.mark.parametrize('name', ['down2', 'up2', 'pad22', 'generic'])
def test_upfirdn2d_oracle_matches_reference(name):
  g = golden('upfirdn2d.npz')
  up, down, p0, p1 = [int(v) for v in g[name + '_p']]
  y = NO.upfirdn2d_native(torch.from_numpy(g[name + '_x']), torch.from_numpy(g[name + '_k']), up=up, down=down, pad=(p0, p1))
  assert y.shape == g[name + '_y'].shape
  assert torch.equal(y, torch.from_numpy(g[name + '_y']))


@pytest.mark.parametrize('name', ['tiny', 'tiny_vp', 'tiny_noattn', 'tiny_ddpmpp', 'tiny_progressive'])
def test_ncsnpp_oracle_matches_reference(name):
  g = golden(f'ncsnpp_{name}.npz')
  cfg = golden_config(name)
  sd = seeded_model(cfg).state_dict()
  taps = {}
  with torch.no_grad():
    y = NO.ncsnpp_forward(sd, cfg, torch.from_numpy(g['x']), torch.from_numpy(g['sigma']), taps=taps)
  stride = int(g.get('tap_stride', 1))       # larger fixtures keep every stride-th element of each image's activation
  for i, v in sorted(taps.items()):
    key = f'tap{i}'
    if key in g:
      assert rel_l2(v.reshape(len(v), -1)[:, ::stride], torch.from_numpy(g[key])) < 2e-6, f'module {i} diverges from the reference'
  assert rel_l2(y, torch.from_numpy(g['y'])) < 2e-6


@pytest.mark.parametrize('name', ['cifar10_ve', 'cifar10_ddpmpp'])
def test_ncsnpp_oracle_matches_reference_cifar10(name):
  g = golden(f'ncsnpp_{name}.npz')
  cfg = golden_config(name)
  sd = seeded_model(cfg).state_dict()
  taps = {}
  with torch.no_grad():
    y = NO.ncsnpp_forward(sd, cfg, torch.from_numpy(g['x']), torch.from_numpy(g['sigma']), taps=taps)
  assert rel_l2(y, torch.from_numpy(g['y'])) < 5e-6
  for i, v in taps.items():
    ref = g['tap_norms'][i]
    if ref > 0:
      assert abs(float(v.double().norm()) - ref) / ref < 5e-6, f'module {i}'


class _OracleModel:
  def __init__(self, cfg):
    self.cfg = cfg
    self.sd = seeded_model(cfg).state_dict()

  def __call__(self, x, labels):
    return NO.ncsnpp_forward(self.sd, self.cfg, x, labels)


def test_pc_sampler_oracle_matches_reference_ve():
  g = golden('pc_ve_tiny.npz')
  cfg = golden_config('tiny')
  model = _OracleModel(cfg)
  shape = tuple(golden('ncsnpp_tiny.npz')['x'].shape)
  sde = SO.VE(0.01, 50, 12)
  torch.manual_seed(11)
  s, nfe = SO.pc_sample(sde, model, shape, 'reverse_diffusion', 'langevin', snr=0.16, n_steps=1, eps=1e-5)
  assert nfe == int(g['nfe'])
  assert rel_l2(s, torch.from_numpy(g['rd_langevin'])) < 1e-5
  torch.manual_seed(12)
  s2, nfe2 = SO.pc_sample(sde, model, shape, 'euler_maruyama', 'none', snr=0.16, n_steps=1, eps=1e-5, denoise=False)
  assert nfe2 == int(g['nfe2'])
  assert rel_l2(s2, torch.from_numpy(g['em_none'])) < 1e-5


def test_pc_sampler_oracle_matches_reference_vp():
  g = golden('pc_vp_tiny.npz')
  cfg = golden_config('tiny_vp')
  model = _OracleModel(cfg)
  shape = tuple(golden('ncsnpp_tiny_vp.npz')['x'].shape)
  sde = SO.VP(0.1, 20., 20)
  torch.manual_seed(21)
  s, _ = SO.pc_sample(sde, model, shape, 'euler_maruyama', 'none', eps=1e-3)
  assert rel_l2(s, torch.from_numpy(g['em_none'])) < 1e-5
  torch.manual_seed(22)
  s, _ = SO.pc_sample(sde, model, shape, 'reverse_diffusion', 'langevin', eps=1e-3)
  assert rel_l2(s, torch.from_numpy(g['rd_langevin'])) < 1e-5


def test_pc_sampler_oracle_matches_reference_none_predictor_and_subvp():
  """Round-2 pins (tools/make_golden_r2.py): a 'none' predictor hands x (not the Langevin mean) to the denoise step;
  the sub-VP SDE under both predictors."""
  g = golden('pc_extra_tiny.npz')
  cfg = golden_config('tiny')
  shape = tuple(golden('ncsnpp_tiny.npz')['x'].shape)
  model = _OracleModel(cfg)        # (re-seeds the generator for its weights: build it before seeding the sampler)
  torch.manual_seed(31)
  s, nfe = SO.pc_sample(SO.VE(0.01, 50, 12), model, shape, 'none', 'langevin', snr=0.16, n_steps=1, eps=1e-5)
  assert nfe == int(g['ve_none_langevin_nfe'])
  assert rel_l2(s, torch.from_numpy(g['ve_none_langevin'])) < 1e-5
  cfg = golden_config('tiny_vp')
  model = _OracleModel(cfg)
  shape = tuple(golden('ncsnpp_tiny_vp.npz')['x'].shape)
  sde = SO.SubVP(0.1, 20., 20)
  torch.manual_seed(32)
  s, _ = SO.pc_sample(sde, model, shape, 'euler_maruyama', 'none', eps=1e-3)
  assert rel_l2(s, torch.from_numpy(g['subvp_em_none'])) < 1e-5
  torch.manual_seed(33)
  s, _ = SO.pc_sample(sde, model, shape, 'reverse_diffusion', 'none', eps=1e-3)
  assert rel_l2(s, torch.from_numpy(g['subvp_rd_none'])) < 1e-5


def test_pc_sampler_oracle_matches_reference_ancestral_and_ald():
  """AncestralSamplingPredictor (sampling.py:204-239) and AnnealedLangevinDynamics (:286-319) under VE and VP
  (tools/make_golden_r2.py, pc_ancestral_ald_tiny.npz)."""
  g = golden('pc_ancestral_ald_tiny.npz')
  model = _OracleModel(golden_config('tiny'))
  shape = tuple(golden('ncsnpp_tiny.npz')['x'].shape)
  torch.manual_seed(34)
  s, _ = SO.pc_sample(SO.VE(0.01, 50, 12), model, shape, 'ancestral_sampling', 'langevin', snr=0.16, n_steps=1, eps=1e-5)
  assert rel_l2(s, torch.from_numpy(g['ve_ancestral_langevin'])) < 1e-5
  torch.manual_seed(35)
  s, _ = SO.pc_sample(SO.VE(0.01, 50, 12), model, shape, 'reverse_diffusion', 'ald', snr=0.16, n_steps=1, eps=1e-5)
  assert rel_l2(s, torch.from_numpy(g['ve_rd_ald'])) < 1e-5
  model = _OracleModel(golden_config('tiny_vp'))
  shape = tuple(golden('ncsnpp_tiny_vp.npz')['x'].shape)
  torch.manual_seed(36)
  s, _ = SO.pc_sample(SO.VP(0.1, 20., 100), model, shape, 'ancestral_sampling', 'ald', snr=0.05, n_steps=1, eps=1e-3)
  assert rel_l2(s, torch.from_numpy(g['vp_ancestral_ald'])) < 1e-5
  torch.manual_seed(37)
  s, _ = SO.pc_sample(SO.VP(0.1, 20., 100), model, shape, 'ancestral_sampling', 'none', snr=0.16, n_steps=1, eps=1e-3)
  assert rel_l2(s, torch.from_numpy(g['vp_ancestral_none'])) < 1e-5


def test_pc_sampler_oracle_matches_reference_ddpmpp():
  """DDPM++ (SURVEY 8 f2; tools/make_golden_ddpmpp.py): the config's own sampler - Euler-Maruyama, no corrector -
  under the VP and sub-VP SDEs, through the reference's get_pc_sampler on the reference's NCSNpp(fir=False,
  embedding_type='positional')."""
  g = golden('pc_ddpmpp_tiny.npz')
  cfg = golden_config('tiny_ddpmpp')
  model = _OracleModel(cfg)
  shape = tuple(golden('ncsnpp_tiny_ddpmpp.npz')['x'].shape)
  torch.manual_seed(41)
  s, nfe = SO.pc_sample(SO.VP(0.1, 20., 20), model, shape, 'euler_maruyama', 'none', eps=1e-3)
  assert nfe == int(g['vp_em_none_nfe'])
  assert rel_l2(s, torch.from_numpy(g['vp_em_none'])) < 1e-5
  torch.manual_seed(42)
  s, _ = SO.pc_sample(SO.SubVP(0.1, 20., 20), model, shape, 'euler_maruyama', 'none', eps=1e-3)
  assert rel_l2(s, torch.from_numpy(g['subvp_em_none'])) < 1e-5


@pytest.mark.parametrize('case', ['ve', 'vp', 'subvp'])
def test_ode_sampler_oracle_matches_reference(case):
  """SURVEY 8 f3 pin (tools/make_golden_ode.py): the reference's get_ode_sampler (scipy RK45, rtol = atol = 1e-5) on the
  reference's own networks; the sub-VP case with the one-step denoise."""
  g = golden('ode_tiny.npz')
  name, sde, eps, denoise = {'ve': ('tiny', SO.VE(0.01, 50, 1000), 1e-5, False),
                             'vp': ('tiny_ddpmpp', SO.VP(0.1, 20., 1000), 1e-3, False),
                             'subvp': ('tiny_ddpmpp', SO.SubVP(0.1, 20., 1000), 1e-3, True)}[case]
  model = _OracleModel(golden_config(name))
  z = torch.from_numpy(g[case + '_z'])
  torch.manual_seed(52)
  s, nfe = SO.ode_sample(sde, model, tuple(z.shape), z=z.clone(), denoise=denoise, eps=eps)
  assert nfe == int(g[case + '_nfe'])
  assert rel_l2(s, torch.from_numpy(g[case])) < 1e-5


def test_sde_tables_match_reference():
  g = golden('sde_tables.npz')
  ve = SO.VE(0.01, 50, 1000)
  t = torch.linspace(1, 1e-5, 1000)
  assert np.array_equal(ve.discretize(torch.zeros(1000, 1, 1, 1), t)[1].numpy(), g['ve_G'])
  assert np.array_equal(ve.sigma(t).numpy(), g['ve_sigma'])
  vp = SO.VP(0.1, 20., 1000)
  t3 = torch.linspace(1, 1e-3, 1000)
  f, G = vp.discretize(torch.ones(1000, 1, 1, 1), t3)
  assert np.array_equal(f.reshape(-1).numpy(), g['vp_f']) and np.array_equal(G.numpy(), g['vp_G'])
  assert np.array_equal(vp.std(t3).numpy(), g['vp_std'])
