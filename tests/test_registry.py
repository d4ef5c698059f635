"""Boundary tests: the reference's registry names / constructor kwargs / state_dict keys (SURVEY §8b, §5) and the model entries
of its config files (stored under tests/golden) loading unchanged. CPU for construction; GPU-marked for forward/train steps."""
import os

import numpy as np
import pytest
import torch

NGP_MODEL = dict(
    type='HashNerfNetwork', cfg=dict(phase='train', chunk=4096, bs_data='rays_o'),
    mlp=dict(type='HashNerfMLP', bound=1,
             embedder_pos=dict(n_input_dims=3, encoding_config=dict(otype='HashGrid', n_levels=16, n_features_per_level=2, log2_hashmap_size=19, base_resolution=16, interpolation='Linear')),
             embedder_dir=dict(n_input_dims=3, encoding_config=dict(otype='SphericalHarmonics', degree=4)),
             density_net=dict(n_input_dims=32, n_output_dims=16, network_config=dict(otype='FullyFusedMLP', activation='ReLU', output_activation='None', n_neurons=64, num_layers=1)),
             color_net=dict(n_output_dims=3, network_config=dict(otype='FullyFusedMLP', activation='ReLU', output_activation='None', n_neurons=64, num_layers=2))),
    sampler=dict(type='NGPGridSampler', update_grid_freq=16, update_block_size=5000000, n_rays_per_batch=4096, cone_angle_constant=0.00390625, near_distance=0.2,
                 target_batch_size=1 << 18, rgb_activation=2, density_activation=3),
    render=dict(type='HashNerfRender', bg_color=[0, 0, 0]))

NERF_MLP = dict(type='NerfMLP', skips=[4], netdepth=8, netwidth=256, netchunk=1024 * 32, output_ch=5, use_viewdirs=True,
                embedder=dict(type='BaseEmbedder', i_embed=0, multires=10, multires_dirs=4))
NERF_MODEL = dict(type='NerfNetwork', cfg=dict(phase='train', N_importance=128, is_perturb=False, chunk=1024 * 32, bs_data='rays_o'), mlp=NERF_MLP, mlp_fine=NERF_MLP,
                  render=dict(type='NerfRender', white_bkgd=True, raw_noise_std=0))
MIP_MODEL = dict(type='MipNerfNetwork', cfg=dict(phase='train', ray_shape='cone', resample_padding=0.01, use_multiscale=False, coarse_loss_mult=0.1, num_levels=2, chunk=800, bs_data='rays_o'),
                 mlp=dict(type='NerfMLP', skips=[4], netdepth=8, netwidth=256, netchunk=1024 * 32, use_viewdirs=True,
                          embedder=dict(type='MipNerfEmbedder', min_deg_point=0, max_deg_point=16, min_deg_view=0, max_deg_view=4, use_viewdirs=True, append_identity=True)),
                 render=dict(type='MipNerfRender', white_bkgd=True, raw_noise_std=0, rgb_padding=0.001, density_bias=-1, density_activation='softplus'))


def test_registry_names_and_state_dict_keys():
    from xrnerf_b200 import registry as R
    for n in ['BaseEmbedder', 'MipNerfEmbedder', 'NerfMLP', 'HashNerfMLP', 'NerfRender', 'MipNerfRender', 'HashNerfRender', 'NGPGridSampler', 'NerfNetwork', 'HashNerfNetwork', 'MipNerfNetwork']:
        assert n in R.MODELS
    net = R.build_network(NGP_MODEL)
    assert sorted(net.state_dict()) == sorted(['sampler.density_grid_bitfield', 'mlp.embedder_pos.params', 'mlp.embedder_dir.params', 'mlp.density_net.params', 'mlp.color_net.params'])
    assert net.state_dict()['mlp.embedder_pos.params'].numel() == 12196240
    assert net.state_dict()['mlp.density_net.params'].numel() == 3072 and net.state_dict()['mlp.color_net.params'].numel() == 7168
    assert len(list(net.parameters())) == 4
    net = R.build_network(NERF_MODEL)
    keys = set(net.state_dict())
    for pre in ('mlp.', 'mlp_fine.'):
        for k in ['pts_linears.0.weight', 'pts_linears.7.bias', 'views_linears.0.weight', 'feature_linear.weight', 'alpha_linear.bias', 'rgb_linear.weight']:
            assert pre + k in keys
    assert net.state_dict()['mlp.pts_linears.5.weight'].shape == (256, 256 + 63)
    assert sum(p.numel() for p in net.mlp.parameters()) == 595844
    mip = R.build_network(MIP_MODEL)
    assert mip.mlp.input_ch == 96 and mip.mlp.input_ch_dirs == 27


def test_reference_config_files_load_unchanged(tmp_path):
    """every config of the three model families: its `model` entry and the last component of its `work_dir` (tests/golden/reference_configs.json, tests/golden/make_golden_host.py)
    written back as a config file, loaded with the '#DATANAME#' substitution and built"""
    import json
    from xrnerf_b200 import registry as R
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_configs.json')) as fh:
        configs = json.load(fh)
    assert len(configs) == 5
    for p, c in configs.items():
        path = tmp_path / os.path.basename(p)
        path.write_text(f'model = {c["model"]!r}\nwork_dir = {c["work_dir"]!r}\n')
        cfg = R.load_config(str(path), dataname='lego')
        assert 'lego' in cfg.work_dir
        net = R.build_network(cfg.model)
        assert type(net).__name__ == c['type'], p


@pytest.mark.gpu
def test_nerf_network_forward_and_train_step_vs_numpy_oracle():
    from oracle import nerf_oracle as O
    from xrnerf_b200 import registry as R
    torch.manual_seed(0)
    small = dict(NERF_MLP, netwidth=64)
    net = R.build_network(dict(NERF_MODEL, mlp=small, mlp_fine=small)).cuda()
    rng = np.random.default_rng(0)
    n, s = 256, 64
    o = (rng.random((n, 3)) * 0.2).astype(np.float32); d = rng.normal(0, 1, (n, 3)).astype(np.float32)
    vd = d / np.linalg.norm(d, axis=-1, keepdims=True)
    z = np.broadcast_to(np.linspace(2, 6, s, dtype=np.float32), (n, s)).copy()
    pts = o[:, None] + d[:, None] * z[..., None]
    data = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in dict(rays_o=o, rays_d=d, viewdirs=vd, z_vals=z, pts=pts, target_s=rng.random((n, 3)).astype(np.float32)).items()}
    with torch.no_grad():
        ret = net.forward(dict(data), is_test=True)
    # oracle chain with the same weights
    sd = {k: v.detach().cpu().numpy() for k, v in net.state_dict().items()}
    raw = O.nerf_mlp(sd, O.embed(pts, vd), 63, 27, prefix='mlp.').reshape(n, s, 4)
    c = O.nerf_render(raw, z, d, white_bkgd=True)
    z2, pts2, _ = O.sample_pdf(z, c['weights'], o, d, 128)
    raw2 = O.nerf_mlp(sd, O.embed(pts2, vd), 63, 27, prefix='mlp_fine.').reshape(n, s + 128, 4)
    f = O.nerf_render(raw2, z2, d, white_bkgd=True)
    assert np.allclose(ret['coarse_rgb'].cpu().numpy(), c['rgb'], atol=2e-4) and np.allclose(ret['rgb'].cpu().numpy(), f['rgb'], atol=5e-4)
    out = net.train_step({k: v[None] for k, v in data.items()}, None)
    assert torch.is_tensor(out['loss']) and out['num_samples'] == n and set(out['log_vars']) == {'loss', 'psnr'}
    out['loss'].backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in net.parameters())


@pytest.mark.gpu
def test_mip_network_forward_and_train_step():
    from xrnerf_b200 import registry as R
    torch.manual_seed(0)
    net = R.build_network(dict(MIP_MODEL, mlp=dict(MIP_MODEL['mlp'], netwidth=64))).cuda()
    rng = np.random.default_rng(1)
    n, s1 = 128, 129
    d = rng.normal(0, 1, (n, 3)).astype(np.float32)
    data = dict(rays_o=(rng.random((n, 3)) * 0.2).astype(np.float32), rays_d=d, viewdirs=d / np.linalg.norm(d, axis=-1, keepdims=True), radii=np.full((n, 1), 1e-3, np.float32),
                lossmult=np.ones((n, 1), np.float32), z_vals=np.broadcast_to(np.linspace(2, 6, s1, dtype=np.float32), (n, s1)).copy(), target_s=rng.random((n, 3)).astype(np.float32))
    data = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in data.items()}
    out = net.train_step({k: v[None] for k, v in data.items()}, None)
    assert set(out['log_vars']) == {'loss', 'loss_fine', 'loss_coarse', 'psnr'}
    out['loss'].backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in net.parameters())


@pytest.mark.gpu
def test_hashnerf_network_train_and_test_steps(scene):
    """the reference's own test (test/models/hashnerf/test_hashnerf_network.py:118) checks isinstance(loss, Tensor); here also: the loss goes down."""
    from xrnerf_b200 import registry as R, synth
    import xrnerf_b200.raymarch_cuda as rm
    torch.manual_seed(0)
    rm.reset_rng()
    net = R.build_network(NGP_MODEL).cuda()
    n_img = scene['poses'].shape[0]
    alldata = dict(poses=scene['poses'], focal=np.full((n_img, 2), synth.FOCAL), aabb_scale=1, aabb_range=(0.0, 1.0), metadata=scene['metadata'])
    net.sampler.set_data(alldata, dict(H=800, W=800))
    opt = torch.optim.Adam(net.parameters(), lr=1e-2, betas=(0.9, 0.99), eps=1e-15)
    n = 4096
    data = dict(rays_o=scene['rays_o'], rays_d=scene['rays_d'], img_ids=scene['img_ids'].astype(np.float32)[:, None], bg_color=np.zeros((n, 3), np.float32),
                alpha=np.ones((n, 1), np.float32), target_s=np.tile(np.array([[0.8, 0.3, 0.1]], np.float32), (n, 1)))
    data = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda()[None] for k, v in data.items()}
    losses = []
    for it in range(12):
        net.sampler.set_iter(it)
        out = net.train_step(dict(data), opt)
        assert torch.is_tensor(out['loss'])
        opt.zero_grad(); out['loss'].backward(); opt.step()
        losses.append(out['log_vars']['loss'])
    assert np.isfinite(losses).all() and losses[-1] < losses[0]
    assert net.sampler.density_grid_bitfield.sum().item() > 0
    with torch.no_grad():
        ret = net.forward({'rays_o': data['rays_o'][0], 'rays_d': data['rays_d'][0], 'img_ids': data['img_ids'][0]}, is_test=True)
    assert ret['rgb'].shape == (n, 3) and ret['alpha'].shape == (n, 1)


@pytest.mark.gpu
def test_fused_nerf_renderer_matches_network_forward():
    """xrnerf_b200.nerf.NerfRenderer (positions + encodings formed inside the kernels, 7 launches) == NerfNetwork.forward(is_test) on the same rays"""
    from xrnerf_b200 import registry as R
    from xrnerf_b200.nerf import NerfRenderer
    torch.manual_seed(0)
    net = R.build_network(NERF_MODEL).cuda()
    rng = np.random.default_rng(0)
    n, s = 700, 64
    o = (rng.random((n, 3)) * 0.2).astype(np.float32); d = rng.normal(0, 1, (n, 3)).astype(np.float32)
    vd = d / np.linalg.norm(d, axis=-1, keepdims=True)
    z = np.broadcast_to(np.linspace(2, 6, s, dtype=np.float32), (n, s)).copy()
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    with torch.no_grad():
        ref = net.forward(dict(rays_o=t(o), rays_d=t(d), viewdirs=t(vd), z_vals=t(z), pts=t(o[:, None] + d[:, None] * z[..., None])), is_test=True)
    out = NerfRenderer(net, near=2.0, far=6.0, n_samples=s).render(t(o), t(d), t(vd))
    assert (out['coarse_rgb'] - ref['coarse_rgb']).abs().max().item() <= 2e-3
    assert (out['rgb'] - ref['rgb']).abs().max().item() <= 5e-3


@pytest.mark.gpu
def test_hashnerf_fused_inference_matches_chunked_forward(scene):
    """HashNerfNetwork.batchify_forward(is_test=True): one fused launch for the whole ray set == the reference-shaped path (sample -> mlp -> render per
    4096-ray chunk) on the same rays, weights, occupancy grid and jitter stream; val_step / test_step keep the reference's keys."""
    from xrnerf_b200 import registry as R, synth
    import xrnerf_b200.raymarch_cuda as rm
    torch.manual_seed(0)
    net = R.build_network(NGP_MODEL).cuda()
    n_img = scene['poses'].shape[0]
    net.sampler.set_data(dict(poses=scene['poses'], focal=np.full((n_img, 2), synth.FOCAL), aabb_scale=1, aabb_range=(0.0, 1.0), metadata=scene['metadata']), dict(H=800, W=800))
    net.sampler.density_grid_bitfield = torch.from_numpy(scene['bitfield']).cuda()
    t, d, c = synth.ngp_weights(seed=3, hash_range=0.5, mlp_gain=2.0)
    with torch.no_grad():
        net.mlp.field.hash_params.copy_(torch.from_numpy(t).cuda()); net.mlp.field.density_params.copy_(torch.from_numpy(d).cuda()); net.mlp.field.color_params.copy_(torch.from_numpy(c).cuda())
    data = {'rays_o': torch.from_numpy(scene['rays_o']).cuda(), 'rays_d': torch.from_numpy(scene['rays_d']).cuda(), 'img_ids': torch.from_numpy(scene['img_ids'].astype(np.float32)[:, None]).cuda()}
    net.chunk, net.bs_data = 4096, 'rays_o'
    with torch.no_grad():
        rm.reset_rng()
        net.fused_inference = False
        ref = net.batchify_forward(dict(data), is_test=True)
        rm.reset_rng()
        net.fused_inference = True
        got = net.batchify_forward(dict(data), is_test=True)
    assert got['rgb'].shape == ref['rgb'].shape == (4096, 3) and got['alpha'].shape == (4096, 1)
    assert (got['rgb'] - ref['rgb']).abs().max().item() <= 2e-3 and (got['alpha'] - ref['alpha']).abs().max().item() <= 2e-3   # fp16 field, fp32 re-association in the scan
    # val_step over two poses through a val pipeline that hands back precomputed rays
    H = W = 64
    def pipeline(item):
        return dict(data, src_shape=torch.tensor([H, W, 3]))
    net.set_val_pipeline(pipeline)
    net.phase = 'train'
    images = torch.rand((2, H, W, 4), device='cuda')
    out = net.val_step({'poses': torch.zeros((1, 2, 4, 3)), 'images': images[None]})
    assert set(out) >= {'rgbs', 'disps', 'gt_imgs', 'elapsed_time', 'psnr'} and len(out['rgbs']) == 2 and out['rgbs'][0].shape == (H, W, 3) and np.isfinite(out['psnr']).all()
    net.phase = 'test'
    sp = net.val_step({'poses': torch.zeros((1, 4, 3)), 'idx': 3})
    assert sp['spiral_rgb'].shape == (H, W, 3) and sp['spiral_alpha'].shape == (H, W, 1) and sp['idx'] == 3
