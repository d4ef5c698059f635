"""Generates the golden data of tests/test_host_utils_vs_reference.py and tests/test_registry.py by running the REFERENCE's own code (imported unmodified
through oracle/ref_import.py, where the reference sources are present) on seeded inputs:

  host_ref_golden.npz       batching.unfold_batching, transforms.recover_shape / merge_ret on seeded tensors (inputs and outputs); the state_dict layout
                            (keys, shapes, input widths) of the reference's NerfMLP for the NeRF and Mip-NeRF embedders, and its first bias under torch.manual_seed(0)
  reference_configs.json    the `model` entry and the last component of `work_dir` of every config file of the three model families, as the config loader returns them

    python tests/golden/make_golden_host.py

The files are committed; the tests only read them.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_import as R  # noqa: E402

UNFOLD_SHAPES = [(1, 7, 3), (2, 5, 3), (3, 4), (6,), (1, 2, 4, 4)]
NERF_MLP_CFGS = [dict(skips=[4], netdepth=8, netwidth=256, output_ch=5, use_viewdirs=True, netchunk=1024 * 32,
                      embedder=dict(type='BaseEmbedder', i_embed=0, multires=10, multires_dirs=4)),
                 dict(skips=[4], netdepth=8, netwidth=256, use_viewdirs=True, netchunk=1024 * 32,
                      embedder=dict(type='MipNerfEmbedder', min_deg_point=0, max_deg_point=16, min_deg_view=0, max_deg_view=4, use_viewdirs=True,
                                    append_identity=True))]
CONFIGS = [('configs/nerf/nerf_blender_base01.py', 'NerfNetwork'), ('configs/nerf/nerf_llff_base01.py', 'NerfNetwork'),
           ('configs/instant_ngp/nerf_blender_local01.py', 'HashNerfNetwork'), ('configs/mipnerf/mipnerf_blender.py', 'MipNerfNetwork'),
           ('configs/mipnerf/mipnerf_multiscale.py', 'MipNerfNetwork')]


def host_utils():
    rb, rt = R.load('networks.utils.batching'), R.load('networks.utils.transforms')
    out = {}
    g = torch.Generator().manual_seed(0)
    for i, shape in enumerate(UNFOLD_SHAPES):
        x = torch.rand(shape, generator=g)
        out[f'unfold.{i}.x'], out[f'unfold.{i}.y'] = x, rb.unfold_batching(x)
    data, sizes = torch.rand((12, 3), generator=g), torch.tensor([3, 4, 3])
    out.update({'recover.data': data, 'recover.sizes': sizes, 'recover.y': rt.recover_shape(data, sizes)})
    a = {k: torch.rand(5, generator=g) for k in ('rgb', 'disp', 'acc')}; b = {k: torch.rand(5, generator=g) for k in ('rgb', 'disp', 'acc')}
    for k in a:
        out[f'merge.a.{k}'], out[f'merge.b.{k}'] = a[k], b[k]
    for k, v in rt.merge_ret(dict(a), dict(b)).items():
        out[f'merge.y.{k}'] = v
    mlpm = R.load('mlps.nerf_mlp'); R.load('embedders.base'); R.load('embedders.mipnerf_embedder')
    for i, cfg in enumerate(NERF_MLP_CFGS):
        torch.manual_seed(0)
        ref = mlpm.NerfMLP(**{k: (dict(v) if isinstance(v, dict) else v) for k, v in cfg.items()})
        sd = ref.state_dict()
        out[f'mlp{i}.keys'] = np.array(list(sd))
        out[f'mlp{i}.shapes'] = np.array([list(v.shape) + [0] * (2 - v.dim()) for v in sd.values()], np.int64)
        out[f'mlp{i}.input_ch'] = np.array([ref.input_ch, ref.input_ch_dirs], np.int64)
        out[f'mlp{i}.pts_linears.0.bias'] = sd['pts_linears.0.bias']
    np.savez_compressed(os.path.join(HERE, 'host_ref_golden.npz'), **{k: (v.numpy() if torch.is_tensor(v) else v) for k, v in out.items()})


def configs():
    from xrnerf_b200 import registry as Reg
    out = {}
    for p, t in CONFIGS:
        cfg = Reg.load_config(os.path.join(R.REF, p))
        # the last component of work_dir carries the '#DATANAME#' placeholder; the directories above it name the authors' machines
        out[p] = {'type': t, 'model': cfg.model, 'work_dir': os.path.basename(os.path.normpath(cfg.work_dir))}
    with open(os.path.join(HERE, 'reference_configs.json'), 'w') as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write('\n')


if __name__ == '__main__':
    assert R.available(), 'the reference sources are not present'
    host_utils()
    configs()
    print('wrote host_ref_golden.npz and reference_configs.json')
