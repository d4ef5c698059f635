"""GPU cross-check against the REFERENCE's own CUDA kernels (extensions/ngp_raymarch built unmodified for sm_100a by oracle/build_ref_cuda.py), through the identical
`raymarch_cuda` signatures. What those kernels computed on a B200 for the inputs below is stored in tests/golden/raymarch_ref_cuda_golden.npz
(tests/golden/make_golden_ref_cuda.py): per-ray sample counts, the samples of a fixed subset of the rays, and the composite of seeded raw values.
The bit-exact contract is defined on the un-contracted CPU build of the same sources (oracle/_ref, tests/test_gpu_raymarch.py): nvcc fuses
the reference's `o + t*d` into FMAs, so here the march may differ in a handful of samples and the tolerances say so."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'raymarch_ref_cuda_golden.npz')
N_COORD_RAYS = 512      # rays whose samples the golden file keeps
BG = (0.1, 0.2, 0.3)


@pytest.fixture(scope='module')
def golden():
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope='module')
def ours():
    import xrnerf_b200.raymarch_cuda as m
    return m


def _march(mod, o, d, bf, cap, ours_mod=None):
    n = o.shape[0]
    md = torch.tensor([[0, 0, 0, 0, .5, .5, 1111., 1111., 0, 0, 0]], dtype=torch.float32, device='cuda')
    xf = torch.zeros((1, 4, 3), dtype=torch.float32, device='cuda'); ids = torch.zeros(n, dtype=torch.int32, device='cuda')
    coords = torch.zeros((cap, 7), dtype=torch.float32, device='cuda'); ridx = torch.zeros((n, 1), dtype=torch.int32, device='cuda')
    ns = torch.zeros((n, 2), dtype=torch.int32, device='cuda'); cnt = torch.zeros(2, dtype=torch.int32, device='cuda')
    if ours_mod is not None:
        ours_mod.reset_rng(ray_sampler=0)
    mod.rays_sampler_api(o, d, bf, md, ids, xf, 0.0, 1.0, 0.05, 1.0 / 256, coords, ridx, ns, cnt)
    torch.cuda.synchronize()
    return coords, ridx, ns, cnt


def scene_rays(scene):
    o = torch.from_numpy(np.ascontiguousarray(scene['rays_o'])).cuda(); d = torch.from_numpy(np.ascontiguousarray(scene['rays_d'])).cuda()
    return o, d, torch.from_numpy(scene['bitfield']).cuda()


def coord_rays(counts):
    """a fixed sample of the rays the reference marched, whose samples are compared one by one"""
    hit = np.nonzero(counts > 0)[0]
    return np.sort(np.random.default_rng(3).choice(hit, min(len(hit), N_COORD_RAYS), replace=False))


def composite_inputs(port, scene):
    """the oracle's march of the scene's rays (bit-exact with ours, tests/test_gpu_raymarch.py) and seeded raw values"""
    n = scene['rays_o'].shape[0]
    c, _, ns, cnt = port.rays_sampler(scene['rays_o'], scene['rays_d'], scene['bitfield'], n * 256)
    raw = (np.random.default_rng(21).standard_normal((int(cnt[1]), 4)) * 0.5).astype(np.float32)
    return raw, np.ascontiguousarray(c[:cnt[1]]), ns


def composite(mod, raw, coords, ns):
    n = ns.shape[0]
    rgb = torch.zeros((n, 3), device='cuda'); alpha = torch.zeros((n, 1), device='cuda')
    mod.calc_rgb_influence_api(torch.from_numpy(raw).cuda(), torch.from_numpy(coords).cuda(), torch.from_numpy(ns).cuda(), torch.tensor(BG), 2, 3, 0.0, 1.0, rgb, alpha)
    torch.cuda.synchronize()
    return rgb.cpu().numpy(), alpha.cpu().numpy()


def test_march_and_composite_agree_with_reference_cuda_kernels(golden, ours, port, scene):
    o, d, bf = scene_rays(scene)
    n = o.shape[0]
    co, _, no, cnto = _march(ours, o, d, bf, n * 256, ours)
    a, b = golden['ns'].astype(np.int64), no[:, 0].cpu().numpy().astype(np.int64)
    assert abs(int(golden['cnt'][1]) - int(cnto[1])) <= max(8, int(cnto[1]) // 2000)
    assert (a != b).mean() < 2e-3                              # per-ray counts: all but FMA-rounding cases
    rays = golden['rays']
    assert np.array_equal(rays, coord_rays(a))
    starts = np.concatenate([[0], np.cumsum(a[rays])])         # the golden samples of the kept rays, ray after ray
    bo, con = no[:, 1].cpu().numpy(), co.cpu().numpy()
    worst, compared = 0.0, 0
    for j, i in enumerate(rays):
        if a[i] == b[i]:
            worst = max(worst, float(np.abs(golden['coords'][starts[j]:starts[j + 1]] - con[bo[i]:bo[i] + a[i]]).max()))
            compared += 1
    assert compared > len(rays) // 2
    assert worst <= 2e-6, worst                                 # positions differ by the FMA's one rounding at most
    # compositing of identical inputs through both kernels
    rgb, alpha = composite(ours, *composite_inputs(port, scene))
    assert float(np.abs(rgb - golden['rgb']).max()) <= 2e-5 and float(np.abs(alpha - golden['alpha']).max()) <= 2e-5
