"""Golden fixtures for the high-resolution NCSN++ family (SURVEY 8 f2: progressive='output_skip',
progressive_input='input_skip', Combine 'sum'; configs/ve/{ffhq,celebahq_256}_ncsnpp_continuous.py) from the REAL
reference, same recipe as tools/make_golden.py.  One small member of the family (three levels, 32x32, FIR resampling): forward at batch 2 with every all_modules[i] activation; plus the state_dict key check of the full-size
CelebA-HQ-256 and FFHQ-1024 configurations (load_state_dict(strict=True) into the reference's constructor, no forward).

    python tools/make_golden_progressive.py
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import make_golden as MG   # noqa: E402
from score_sde_pytorch_b200 import configs as our_configs   # noqa: E402


def progressive_configs():
  # (fir=False cannot be pinned: the reference's Upsample(fir=False) calls F.interpolate(x, (2H, 2W), 'nearest') with the
  # mode in the scale_factor slot (layerspp.py:116), which current PyTorch rejects - a reference quirk, not reproduced)
  return {'tiny_progressive': (our_configs.tiny_progressive(), 2)}


def main():
  torch.set_num_threads(8)
  sde_lib, sampling, ncsnpp, mutils, _ = MG.import_reference()
  for name, (cfg, B) in progressive_configs().items():
    cfg.device = torch.device('cpu')
    sd = MG.our_weights(cfg)
    torch.manual_seed(0)
    ref_model = mutils.get_model('ncsnpp')(cfg).eval()
    ref_model.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(7)
    R, C = cfg.data.image_size, cfg.data.num_channels
    x = torch.randn(B, C, R, R, generator=g) * 3.0
    sigma = torch.exp(torch.linspace(np.log(40.0), np.log(0.02), B))
    with torch.no_grad():
      y = ref_model(x, sigma)
      taps, hooks = {}, []
      for i, mod in enumerate(ref_model.all_modules):
        hooks.append(mod.register_forward_hook(lambda m, a, o, i=i: taps.__setitem__(i, o.detach().clone())))
      ref_model(x, sigma)
      for h in hooks:
        h.remove()
    # every third element of each image's activation keeps the fixture under 1 MB (tests/test_oracle_golden.py reads tap_stride)
    rec = dict(x=x.numpy(), sigma=sigma.numpy(), y=y.numpy(), tap_stride=np.array(3))
    for i, v in taps.items():
      rec[f'tap{i}'] = np.ascontiguousarray(v.reshape(B, -1)[:, ::3].numpy())
    np.savez_compressed(os.path.join(MG.OUT, f'ncsnpp_{name}.npz'), **rec)
    print(name, 'forward done', float(y.abs().mean()), 'modules', len(ref_model.all_modules))
  # full-size members: key / shape layout only (the 1024x1024 forward is a GPU job)
  for nm, cfg in (('celebahq_256', our_configs.ve_celebahq_256_ncsnpp_continuous()), ('ffhq_1024', our_configs.ve_ffhq_1024_ncsnpp_continuous())):
    cfg.device = torch.device('cpu')
    sd = MG.our_weights(cfg)
    ref_model = mutils.get_model('ncsnpp')(cfg)
    ref_model.load_state_dict(sd, strict=True)
    print(nm, 'state_dict layout matches the reference:', len(sd), 'tensors,', sum(v.numel() for k, v in sd.items() if k != 'sigmas'), 'parameters')


if __name__ == '__main__':
  main()
