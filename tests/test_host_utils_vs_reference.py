"""Host-side helpers of the networks against the REFERENCE's own functions: batching.unfold_batching, transforms.recover_shape / merge_ret
(networks/utils/batching.py:5-12, transforms.py:5-31), and NGPGridSampler.update_batch_rays (samplers/ngp_grid_sampler.py:268-284, restated: the reference
class imports its CUDA extension at module import). The reference's outputs are stored in tests/golden/host_ref_golden.npz (tests/golden/make_golden_host.py)."""
import math
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'host_ref_golden.npz')
N_UNFOLD = 5


@pytest.fixture(scope='module')
def golden():
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


def test_unfold_batching_recover_shape_merge_ret_match_reference(golden):
    from xrnerf_b200.registry import networks as N
    G = {k: torch.from_numpy(v) for k, v in golden.items() if v.dtype.kind != 'U'}
    for i in range(N_UNFOLD):
        assert torch.equal(N.unfold_batching(G[f'unfold.{i}.x']), G[f'unfold.{i}.y']), G[f'unfold.{i}.x'].shape
    assert torch.equal(N.recover_shape(G['recover.data'], G['recover.sizes']), G['recover.y'])
    keys = ('rgb', 'disp', 'acc')
    ours = N.merge_ret({k: G[f'merge.a.{k}'] for k in keys}, {k: G[f'merge.b.{k}'] for k in keys})
    assert set(ours) == {k[len('merge.y.'):] for k in G if k.startswith('merge.y.')}
    assert all(torch.equal(v, G['merge.y.' + k]) for k, v in ours.items())


def test_update_batch_rays_rule():
    """n_rays <- min(ceil128(int(n_rays * 2^18 / max(measured / 16, 1))), 2^18), every update_grid_freq-th step, then the counter is cleared."""
    from xrnerf_b200 import registry as R
    smp = R.build_sampler(dict(type='NGPGridSampler', update_grid_freq=16, update_block_size=5000000, n_rays_per_batch=4096, cone_angle_constant=0.00390625, near_distance=0.2,
                               target_batch_size=1 << 18, rgb_activation=2, density_activation=3))
    for measured, n0 in [(16 * 40000, 4096), (16 * 300000, 65536), (0, 4096), (16 * 262144, 262144)]:
        smp.n_rays_per_batch = n0
        smp.measured_batch_size = torch.tensor([measured], dtype=torch.int32)
        smp.set_iter(15)
        smp.update_batch_rays(True)
        m = max(measured / 16, 1)
        want = int(min(math.ceil(int(n0 * (1 << 18) / m) / 128) * 128, 1 << 18))
        assert smp.n_rays_per_batch == want and smp.measured_batch_size.item() == 0
        smp.n_rays_per_batch = n0
        smp.measured_batch_size = torch.tensor([measured], dtype=torch.int32)
        smp.set_iter(14)
        smp.update_batch_rays(True)
        assert smp.n_rays_per_batch == n0 and smp.measured_batch_size.item() == measured


def test_reference_nerf_mlp_checkpoints_load_into_registry_modules(golden):
    """SURVEY 8f-4 (checkpoint compatibility): a state_dict laid out as the REFERENCE's own NerfMLP's (NeRF and Mip-NeRF embedders: keys in order, shapes,
    input widths, as stored in the golden file) has exactly our keys and shapes and loads with strict=True; the packed tcgen05 weight image is rebuilt
    from the loaded weights."""
    from xrnerf_b200 import registry as R
    from xrnerf_b200.nerf_mlp import pack_nerf_mlp_v3
    cfgs = [dict(skips=[4], netdepth=8, netwidth=256, output_ch=5, use_viewdirs=True, netchunk=1024 * 32, embedder=dict(type='BaseEmbedder', i_embed=0, multires=10, multires_dirs=4)),
            dict(skips=[4], netdepth=8, netwidth=256, use_viewdirs=True, netchunk=1024 * 32,
                 embedder=dict(type='MipNerfEmbedder', min_deg_point=0, max_deg_point=16, min_deg_view=0, max_deg_view=4, use_viewdirs=True, append_identity=True))]
    for i, cfg in enumerate(cfgs):
        g = torch.Generator().manual_seed(i)
        sd_ref = {}
        for k, shape in zip(golden[f'mlp{i}.keys'].tolist(), golden[f'mlp{i}.shapes'].tolist()):
            sd_ref[k] = torch.randn([s for s in shape if s], generator=g) * 0.05
        sd_ref['pts_linears.0.bias'] = torch.from_numpy(golden[f'mlp{i}.pts_linears.0.bias'])
        ours = R.build_mlp(dict(cfg, type='NerfMLP'))
        sd_ours = ours.state_dict()
        assert list(sd_ref) == list(sd_ours) and all(sd_ref[k].shape == sd_ours[k].shape for k in sd_ref)
        assert (ours.input_ch, ours.input_ch_dirs) == tuple(golden[f'mlp{i}.input_ch'].tolist())
        ours.load_state_dict(sd_ref, strict=True)
        image, bias = pack_nerf_mlp_v3(ours)
        assert torch.equal(bias[:256], sd_ref['pts_linears.0.bias']) and image.numel() > 1_000_000
