"""CPU tests of the host-side mirror of the reference surface (sampling / sde_lib /
models.utils), of the schedule tables handed to the native loop, and of the C-ABI library
(loads, exports every declared symbol; no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from helpers import golden, golden_config, seeded_model, rel_l2
from oracle import ncsnpp_oracle as NO
from score_sde_pytorch_b200 import _lib, configs, native, sampling, sde_lib
from score_sde_pytorch_b200.models import utils as mutils

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class TorchModel(torch.nn.Module):
  """A user-style nn.Module score model (oracle arithmetic) to drive the generic host loop."""

  def __init__(self, cfg):
    super().__init__()
    self.cfg = cfg
    self.sd = seeded_model(cfg).state_dict()

  def forward(self, x, labels):
    return NO.ncsnpp_forward(self.sd, self.cfg, x, labels)


def test_generic_pc_loop_matches_reference_ve():
  g = golden('pc_ve_tiny.npz')
  cfg = golden_config('tiny')
  cfg.device = torch.device('cpu')
  model = TorchModel(cfg)
  shape = tuple(golden('ncsnpp_tiny.npz')['x'].shape)
  sde = sde_lib.VESDE(0.01, 50, 12)
  fn = sampling.get_pc_sampler(sde, shape, sampling.ReverseDiffusionPredictor, sampling.LangevinCorrector,
                               lambda v: v, snr=0.16, n_steps=1, continuous=True, denoise=True, eps=1e-5, device='cpu')
  torch.manual_seed(11)
  s, nfe = fn(model)
  assert nfe == int(g['nfe']) == 24
  assert rel_l2(s, torch.from_numpy(g['rd_langevin'])) < 1e-5


def test_get_sampling_fn_vp_em_plumbing():
  """BASELINE.json configs[0]-style plumbing: VP SDE, Euler-Maruyama predictor only, 20 steps, B=2, CPU."""
  g = golden('pc_vp_tiny.npz')
  cfg = golden_config('tiny_vp')
  cfg.device = torch.device('cpu')
  cfg.sampling.predictor, cfg.sampling.corrector = 'euler_maruyama', 'none'
  model = TorchModel(cfg)
  shape = tuple(golden('ncsnpp_tiny_vp.npz')['x'].shape)
  sde = sde_lib.VPSDE(0.1, 20., 20)
  fn = sampling.get_sampling_fn(cfg, sde, shape, lambda v: v, 1e-3)
  torch.manual_seed(21)
  s, nfe = fn(model)
  assert nfe == 40          # N*(n_steps+1) even with the None corrector (sampling.py:409)
  assert rel_l2(s, torch.from_numpy(g['em_none'])) < 1e-5
  cfg.sampling.predictor, cfg.sampling.corrector = 'reverse_diffusion', 'langevin'
  fn = sampling.get_sampling_fn(cfg, sde, shape, lambda v: v, 1e-3)
  torch.manual_seed(22)
  s, _ = fn(model)
  assert rel_l2(s, torch.from_numpy(g['rd_langevin'])) < 1e-5


def test_generic_pc_loop_none_predictor_and_subvp_match_reference():
  """Host mirror (generic loop) vs the round-2 reference goldens: predictor=None hands the noisy state to the denoise
  step (sampling.py:241-250); sub-VP under both predictors."""
  g = golden('pc_extra_tiny.npz')
  cfg = golden_config('tiny')
  cfg.device = torch.device('cpu')
  model = TorchModel(cfg)
  shape = tuple(golden('ncsnpp_tiny.npz')['x'].shape)
  fn = sampling.get_pc_sampler(sde_lib.VESDE(0.01, 50, 12), shape, None, sampling.LangevinCorrector, lambda v: v, snr=0.16,
                               n_steps=1, continuous=True, denoise=True, eps=1e-5, device='cpu')
  torch.manual_seed(31)
  s, nfe = fn(model)
  assert nfe == int(g['ve_none_langevin_nfe'])
  assert rel_l2(s, torch.from_numpy(g['ve_none_langevin'])) < 1e-5
  cfg = golden_config('tiny_vp')
  cfg.device = torch.device('cpu')
  model = TorchModel(cfg)
  shape = tuple(golden('ncsnpp_tiny_vp.npz')['x'].shape)
  sde = sde_lib.subVPSDE(0.1, 20., 20)
  for tag, pred, seed in (('subvp_em_none', sampling.EulerMaruyamaPredictor, 32), ('subvp_rd_none', sampling.ReverseDiffusionPredictor, 33)):
    fn = sampling.get_pc_sampler(sde, shape, pred, sampling.NoneCorrector, lambda v: v, snr=0.16, n_steps=1,
                                 continuous=True, denoise=True, eps=1e-3, device='cpu')
    torch.manual_seed(seed)
    s, _ = fn(model)
    assert rel_l2(s, torch.from_numpy(g[tag])) < 1e-5, tag


def test_registries_and_errors():
  assert sampling.get_predictor('reverse_diffusion') is sampling.ReverseDiffusionPredictor
  assert sampling.get_corrector('langevin') is sampling.LangevinCorrector
  assert set(sampling._PREDICTORS) >= {'euler_maruyama', 'reverse_diffusion', 'ancestral_sampling', 'none'}
  assert set(sampling._CORRECTORS) >= {'langevin', 'ald', 'none'}
  with pytest.raises(ValueError):
    sampling.register_predictor(name='none')(sampling.NonePredictor)
  with pytest.raises(ValueError):
    mutils.register_model(name='ncsnpp')(object)

  @sampling.register_corrector
  class MyCorrector(sampling.Corrector):
    def update_fn(self, x, t):
      return x, x
  assert sampling.get_corrector('MyCorrector') is MyCorrector
  del sampling._CORRECTORS['MyCorrector']

  cfg = configs.ve_cifar10_ncsnpp_continuous()
  cfg.sampling.method = 'bogus'
  with pytest.raises(ValueError):
    sampling.get_sampling_fn(cfg, sde_lib.VESDE(), (1, 3, 32, 32), lambda v: v, 1e-5)

  class OtherSDE(sde_lib.SDE):
    T = 1
    def sde(self, x, t): return x, t
    def marginal_prob(self, x, t): return x, t
    def prior_sampling(self, shape): return torch.zeros(*shape)
    def prior_logp(self, z): return z
  with pytest.raises(NotImplementedError):
    mutils.get_score_fn(OtherSDE(10), lambda x, t: x)
  with pytest.raises(NotImplementedError):
    sampling.LangevinCorrector(OtherSDE(10), None, 0.1, 1)


def test_schedule_tables_match_reference_scalars():
  g = golden('sde_tables.npz')
  tb = native.build_tables(sde_lib.VESDE(0.01, 50, 1000), 'reverse_diffusion', 'langevin', False, 1e-5)
  assert np.array_equal(tb['label'], g['ve_sigma'])
  assert np.array_equal(tb['pc'], g['ve_G'])
  assert np.allclose(tb['pb'], g['ve_G'] ** 2, rtol=1e-6)
  vp = native.build_tables(sde_lib.VPSDE(0.1, 20., 1000), 'reverse_diffusion', 'langevin', False, 1e-3)
  assert np.array_equal(vp['pc'], g['vp_G'])
  # x_mean = x - f - ... with x = 1: pa = 1 - f
  assert np.allclose(vp['pa'], 1.0 - g['vp_f'], rtol=1e-6)
  assert np.allclose(vp['score_scale'], -1.0 / g['vp_std'], rtol=1e-6)


def test_affine_predictor_tables_reproduce_host_predictors():
  """The (pa, pb, pc) tables must reproduce the class-based predictors for arbitrary network outputs."""
  torch.manual_seed(0)
  x = torch.randn(3, 2, 4, 4)
  out = torch.randn(3, 2, 4, 4)
  z = torch.randn(3, 2, 4, 4)
  for sde, eps in ((sde_lib.VESDE(0.01, 50, 50), 1e-5), (sde_lib.VPSDE(0.1, 20., 50), 1e-3), (sde_lib.subVPSDE(0.1, 20., 50), 1e-3)):
    for kind, cls in (('reverse_diffusion', sampling.ReverseDiffusionPredictor), ('euler_maruyama', sampling.EulerMaruyamaPredictor)):
      for pf in (False, True):
        if pf and kind == 'euler_maruyama':
          continue   # the reference's EM predictor cannot run with probability_flow (float diffusion is indexed, sampling.py:186)
        tb = native.build_tables(sde, kind, 'none', pf, eps)
        ts = torch.linspace(sde.T, eps, sde.N)
        for i in (0, 7, sde.N - 1):
          t = torch.ones(3) * ts[i]
          score_fn = mutils.get_score_fn(sde, torch.nn.Identity(), train=False, continuous=True)
          score_fn._model_fn = lambda xx, labels: out      # fixed "network output"
          pred = cls(sde, score_fn, pf)
          torch.manual_seed(5)
          xn, xm = pred.update_fn(x, t)
          torch.manual_seed(5)
          zz = torch.randn_like(x)
          xm2 = float(tb['pa'][i]) * x + float(tb['pb'][i]) * out
          xn2 = xm2 + float(tb['pc'][i]) * zz
          assert torch.allclose(xm, xm2, rtol=2e-5, atol=2e-5), (type(sde).__name__, kind, pf, i)
          assert torch.allclose(xn, xn2, rtol=2e-5, atol=2e-5), (type(sde).__name__, kind, pf, i)


def test_affine_tables_reproduce_ancestral_sampling_and_annealed_langevin():
  """Round 2: AncestralSamplingPredictor (sampling.py:204-239) and AnnealedLangevinDynamics (:286-319) are affine in
  (x, network output, noise) too, so the native loop runs them from tables; the tables must reproduce the classes."""
  class Fixed(torch.nn.Module):
    def __init__(self, out):
      super().__init__()
      self.out = out

    def forward(self, x, labels):
      return self.out

  torch.manual_seed(0)
  x, out = torch.randn(3, 2, 4, 4), torch.randn(3, 2, 4, 4)
  for sde, eps in ((sde_lib.VESDE(0.01, 50, 50), 1e-5), (sde_lib.VPSDE(0.1, 20., 50), 1e-3)):
    score_fn = mutils.get_score_fn(sde, Fixed(out), train=False, continuous=True)
    tb = native.build_tables(sde, 'ancestral_sampling', 'ald', False, eps, snr=0.17)
    ts = torch.linspace(sde.T, eps, sde.N)
    for i in (0, 7, sde.N - 1):
      t = torch.ones(3) * ts[i]
      torch.manual_seed(5)
      xn, xm = sampling.AncestralSamplingPredictor(sde, score_fn, False).update_fn(x, t)
      torch.manual_seed(5)
      zz = torch.randn_like(x)
      xm2 = float(tb['pa'][i]) * x + float(tb['pb'][i]) * out
      assert torch.allclose(xm, xm2, rtol=2e-5, atol=2e-5) and torch.allclose(xn, xm2 + float(tb['pc'][i]) * zz, rtol=2e-5, atol=2e-5)
      torch.manual_seed(6)
      xn, xm = sampling.AnnealedLangevinDynamics(sde, score_fn, 0.17, 1).update_fn(x, t)
      torch.manual_seed(6)
      zz = torch.randn_like(x)
      xm2 = float(tb['ca'][i]) * x + float(tb['cb'][i]) * out
      assert torch.allclose(xm, xm2, rtol=2e-5, atol=2e-5) and torch.allclose(xn, xm2 + float(tb['cc'][i]) * zz, rtol=2e-5, atol=2e-5)
  # combinations the reference itself rejects stay on the host loop (which raises like the reference)
  m = seeded_model(golden_config('tiny'))
  kw = dict(shape=(2, 3, 16, 16), snr=0.16, n_steps=1, continuous=True, eps=1e-3, device='cuda')
  assert native.match_pc_plan(sde=sde_lib.subVPSDE(0.1, 20., 10), model=m, predictor=sampling.AncestralSamplingPredictor,
                              corrector=sampling.NoneCorrector, probability_flow=False, **kw) is None


def test_library_loads_and_exports_every_declared_symbol():
  lib = _lib.load()
  assert lib.b200_version() >= 100
  header = open(os.path.join(REPO, 'include', 'scoresde_b200.h')).read()
  declared = set(re.findall(r'B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(', header))
  assert declared, 'no declarations parsed'
  for name in declared:
    assert hasattr(lib, name), f'{name} declared in the header but not exported'
  assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
  err = lib.b200_last_error()
  assert isinstance(err, bytes)


def test_engine_param_table_matches_module_and_reference_names():
  for name in ('tiny', 'tiny_noattn', 'cifar10_ve'):
    cfg = golden_config(name)
    m = seeded_model(cfg)
    table = m.native_param_table()
    sd = dict(m.named_parameters())
    assert [n for n, _ in table if n not in sd] == []
    assert sorted(n for n, _ in table) == sorted(sd)
    for n, shape in table:
      assert tuple(sd[n].shape) == shape
  assert sum(p.numel() for p in seeded_model(golden_config('cifar10_ve')).parameters()) == 62758915


def test_ddpmpp_engine_param_table_has_the_reference_names_plus_the_frequency_table():
  """DDPM++ (fir=False, positional embedding, no pyramid): the positional embedding has no module in the reference's
  all_modules (ncsnpp.py:79-83), so every later index is one lower than in the Fourier family; the engine's only extra
  input is the frequency table, which is NOT a state_dict key (non-persistent buffer built with the reference's ops)."""
  import math
  for name in ('tiny_ddpmpp', 'cifar10_ddpmpp'):
    cfg = golden_config(name)
    m = seeded_model(cfg)
    table = m.native_param_table()
    sd = dict(m.named_parameters())
    assert table[0][0] == 'pos_freqs' and table[0][1] == (cfg.model.nf // 2,)
    assert sorted(n for n, _ in table[1:]) == sorted(sd)
    for n, shape in table[1:]:
      assert tuple(sd[n].shape) == shape
    assert 'pos_freqs' not in m.state_dict() and 'all_modules.0.weight' in sd and sd['all_modules.0.weight'].shape[1] == cfg.model.nf
    half = cfg.model.nf // 2
    want = torch.exp(torch.arange(half, dtype=torch.float32) * -(math.log(10000) / (half - 1)))
    assert torch.equal(m.pos_freqs, want)
  cfg = golden_config('tiny_ddpmpp')
  cfg.model.scale_by_sigma = True          # would need sigmas[time_cond.long()] (ncsnpp.py:245): not supported, must say so
  with pytest.raises(NotImplementedError):
    seeded_model(cfg)


def test_progressive_family_param_tables_match_module():
  """output_skip / input_skip (SURVEY 8 f2): engine parameter table == module parameters for a small member and for the
  full-size CelebA-HQ-256 / FFHQ-1024 configurations (whose state_dict layouts tools/make_golden_progressive.py loads
  into the reference's constructor with strict=True: 65 574 549 and 105 785 896 parameters)."""
  for name, nparams in (('tiny_progressive', None), ('celebahq_256', 65574549), ('ffhq_1024', 105785896)):
    cfg = golden_config(name)
    m = seeded_model(cfg)
    table = m.native_param_table()
    sd = dict(m.named_parameters())
    assert sorted(n for n, _ in table) == sorted(sd), name
    for n, shape in table:
      assert tuple(sd[n].shape) == shape
    if nparams:
      assert sum(p.numel() for p in m.parameters()) == nparams
  cfg = golden_config('tiny_progressive')
  cfg.model.progressive_combine = 'cat'
  with pytest.raises(NotImplementedError):
    seeded_model(cfg)
  cfg = golden_config('tiny_progressive')
  cfg.model.progressive = 'residual'
  with pytest.raises(NotImplementedError):
    seeded_model(cfg)


def test_product_model_has_no_cpu_path():
  m = seeded_model(golden_config('tiny'))
  with pytest.raises(RuntimeError, match='CUDA'):
    m(torch.zeros(1, 3, 16, 16), torch.ones(1))
  cfg = golden_config('tiny')
  cfg.model.resblock_type = 'ddpm'
  with pytest.raises(NotImplementedError):
    seeded_model(cfg)


def test_bench_reference_arm_prints_the_contract_line(tmp_path):
  """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): one JSON line with the same
  metric/unit/config keys, `impl: reference`, a cpu_baseline describing the run and a zero-copy e2e block."""
  import json
  import os
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  env = dict(os.environ, OMP_NUM_THREADS='1')      # what torchrun exports to every rank
  out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '5', '--warmup', '0',
                        '--cpu-batch', '1', '--dump-outputs', str(tmp_path / 'out')], capture_output=True, text=True, timeout=900, env=env, cwd=root)
  assert out.returncode == 0, out.stderr[-2000:]
  line = json.loads(out.stdout.strip().splitlines()[-1])
  assert line['impl'] == 'reference' and line['unit'] == 'images/s' and line['higher_is_better'] is True
  assert line['metric'].startswith('PC-sampler images/sec') and line['value'] > 0 and line['n_gpus'] == 1
  cb = line['cpu_baseline']
  # the UNMODIFIED reference from baseline/_ref (tools/install_ref.sh) when it is installed, else the oracle port
  want = 'reference' if os.path.isdir(os.path.join(root, 'baseline', '_ref', 'models')) else 'port'
  assert cb['kind'] == want and cb['value'] == line['value'] and cb['cores'] >= 1 and 'PC iterations' in cb['sample']
  assert line['steps'] == 5 and len(cb['iter_seconds']) == 5      # --steps sets the timed iterations; their median is reported
  assert line['e2e'] == {'value': line['value'], 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
  if (os.cpu_count() or 1) >= 4:
    assert cb['cores'] > 1        # OMP_NUM_THREADS=1 from the launcher must not reduce the arm to one core
  import numpy as np
  for name in ('x', 'x_mean'):    # the state the last timed PC iteration returned
    a = np.load(tmp_path / 'out' / f'{name}.npy')
    assert a.dtype == np.float32 and a.shape == (1, 3, 32, 32) and np.isfinite(a).all()


def test_bench_dump_outputs_keeps_a_fixed_sample_under_the_size_limit(tmp_path, monkeypatch):
  import os
  import sys
  import numpy as np
  sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
  import bench
  x = torch.arange(10 * 6, dtype=torch.float32).reshape(10, 2, 3)
  xm = x.double() * 2
  bench.dump_outputs(str(tmp_path / 'all'), dict(x=x, x_mean=xm))
  assert np.array_equal(np.load(tmp_path / 'all' / 'x.npy'), x.numpy())
  assert np.load(tmp_path / 'all' / 'x_mean.npy').dtype == np.float64
  monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 4 * (6 * 4 + 6 * 8))     # room for four images of both arrays
  for d in ('a', 'b'):
    bench.dump_outputs(str(tmp_path / d), dict(x=x, x_mean=xm))
  a, am = np.load(tmp_path / 'a' / 'x.npy'), np.load(tmp_path / 'a' / 'x_mean.npy')
  assert a.shape == (4, 2, 3) and np.array_equal(am, a.astype(np.float64) * 2)   # the same images of every array
  assert np.array_equal(a, np.load(tmp_path / 'b' / 'x.npy'))                   # the same images on every run


def test_ema_matches_reference_update_rule_and_notifies_the_engine_module(tmp_path):
  """models/ema.py:34-51 semantics (decay ramp min(decay, (1+n)/(10+n)), positional shadow list over the trainable
  parameters), checkpoint round trip in the reference's file format (utils.py:7-30), and the engine hook: copy_to /
  restore bump the owning NCSNpp's weight version so the packed device copy is rebuilt."""
  from score_sde_pytorch_b200 import utils as butils
  from score_sde_pytorch_b200.models.ema import ExponentialMovingAverage
  from score_sde_pytorch_b200.models.ncsnpp import NCSNpp
  cfg = golden_config('tiny')
  torch.manual_seed(0)
  model = NCSNpp(cfg)
  params = list(model.parameters())
  trainable = [p for p in params if p.requires_grad]
  assert len(trainable) == len(params) - 1          # the Fourier projection W is frozen, as in the reference
  ema = ExponentialMovingAverage(params, decay=0.999)
  assert len(ema.shadow_params) == len(trainable)
  start = [p.detach().clone() for p in trainable]
  with torch.no_grad():
    for p in trainable:
      p.add_(1.0)
  ema.update(params)                                # n = 1: decay = min(0.999, 2/11)
  d = 2.0 / 11.0
  for s, p0 in zip(ema.shadow_params, start):
    assert torch.allclose(s, p0 + (1.0 - d), atol=1e-6)
  ema.update(params)                                # n = 2: decay = 3/12
  d2 = 3.0 / 12.0
  for s, p0 in zip(ema.shadow_params, start):
    assert torch.allclose(s, p0 + 1.0 - d2 * d, atol=1e-6)
  with pytest.raises(ValueError):
    ExponentialMovingAverage(params, decay=1.5)
  # store / copy_to / restore, each notifying the engine-backed module
  v0 = model._weights_version
  ema.store(params)
  ema.copy_to(params)
  assert model._weights_version == v0 + 1
  assert all(torch.equal(p, s) for p, s in zip(trainable, ema.shadow_params))
  ema.restore(params)
  assert model._weights_version == v0 + 2
  assert all(torch.allclose(p, p0 + 1.0) for p, p0 in zip(trainable, start))
  # checkpoint round trip in the reference's format
  path = str(tmp_path / 'ckpt' / 'checkpoint_1.pth')
  state = dict(optimizer=torch.optim.Adam(model.parameters(), lr=1e-3), model=model, ema=ema, step=7)
  assert butils.restore_checkpoint(path, state, 'cpu') is state          # missing file: unchanged state, directory created
  butils.save_checkpoint(path, state)
  torch.manual_seed(1)
  model2 = NCSNpp(cfg)
  ema2 = ExponentialMovingAverage(model2.parameters(), decay=0.5)
  state2 = butils.restore_checkpoint(path, dict(optimizer=None, model=model2, ema=ema2, step=0), 'cpu')
  assert state2['step'] == 7 and ema2.decay == 0.999 and ema2.num_updates == 2
  assert all(torch.equal(a, b) for a, b in zip(model2.state_dict().values(), model.state_dict().values()))
  assert all(torch.equal(a, b) for a, b in zip(ema2.shadow_params, ema.shadow_params))
  # a DataParallel-era checkpoint (keys prefixed with 'module.') loads too
  torch.save({'optimizer': {}, 'model': {'module.' + k: v for k, v in model.state_dict().items()}, 'ema': ema.state_dict(), 'step': 3}, path)
  state3 = butils.restore_checkpoint(path, dict(optimizer=None, model=model2, ema=ema2, step=0), 'cpu')
  assert state3['step'] == 3


@pytest.mark.parametrize('name', ['tiny', 'tiny_noattn', 'cifar10_ve'])
def test_parameter_list_matches_the_reference_order(name):
  """EMA shadow parameters in reference checkpoints are positional (models/ema.py:27-28): same names, shapes and
  requires_grad flags in the same `parameters()` order as the reference's NCSNpp (tools/make_param_order.py)."""
  import json
  import os
  ref = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'param_order.json')))[name]
  model = seeded_model(golden_config(name))
  mine = [[n, list(p.shape), bool(p.requires_grad)] for n, p in model.named_parameters()]
  assert mine == ref


def test_profile_tooling_reads_the_committed_artifacts():
  """The roofline block of bench.py takes `traffic` from profiles/traffic_f16.json (written by
  tools/summarize_traffic.py from an ncu metrics pass); the launch-list summariser must keep parsing the committed CSV."""
  import glob
  import os
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  sys.path.insert(0, root)
  import bench
  t = bench.load_traffic('f16')
  assert isinstance(t, int) and t > 10_000_000            # DRAM bytes per contraction launch
  assert bench.load_traffic('no-such-precision') is None
  csvs = sorted(glob.glob(os.path.join(root, 'profiles', '*launches_pc_step*_f16.csv')))
  assert csvs, 'no committed launch list'
  out = subprocess.run([sys.executable, os.path.join(root, 'tools', 'summarize_launches.py'), csvs[-1]],
                       capture_output=True, text=True, timeout=120)
  assert out.returncode == 0 and 'gemm_tc' in out.stdout and 'gn_apply' in out.stdout


def test_execution_options_reach_the_native_config():
  """Per-engine options are fields of b200_ncsnpp_config (nothing is read from the environment).  `halo`: the package
  default is the halo form in the swapped AND the CTA-pair kernel (no_halo = 2); True / False / raw ints map as documented
  in include/scoresde_b200.h."""
  from score_sde_pytorch_b200.models.ncsnpp import NCSNpp
  cfg = golden_config('tiny')
  want = {None: 2, 'pairs': 2, True: 0, False: 1, 2 | 8: 10, 6: 6}
  for halo, no_halo in want.items():
    m = NCSNpp(cfg) if halo is None else NCSNpp(cfg, halo=halo)
    assert m._native_config().no_halo == no_halo, (halo, m._native_config().no_halo)
  c = NCSNpp(cfg, precision='f16', separate_groupnorm=False, pdl=True, cuda_core_head=True)._native_config()
  assert (c.precision, c.separate_groupnorm, c.pdl, c.cuda_core_head) == (2, 0, 1, 1)
