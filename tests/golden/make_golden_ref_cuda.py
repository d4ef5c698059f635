"""Generates tests/golden/raymarch_ref_cuda_golden.npz: the REFERENCE's own `raymarch_cuda` kernels (oracle/_ref/cuda, built by oracle/build_ref_cuda.py where
the reference sources are present) run on a B200 on the inputs of tests/test_gpu_vs_ref_cuda.py.

    python tests/golden/make_golden_ref_cuda.py [OUT.npz]

The .npz is committed; the test only reads it.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
from oracle import build_ref_cuda  # noqa: E402
from oracle.oracle import Port  # noqa: E402
from xrnerf_b200 import synth  # noqa: E402
import test_gpu_vs_ref_cuda as T  # noqa: E402


def main(out_path):
    import torch
    ref = build_ref_cuda.load_module()
    assert ref is not None, 'oracle/_ref/cuda/raymarch_cuda_ref.so is not built'
    torch.cuda.set_device(0)
    grid = synth.lego_like_density_grid(0)       # the `scene` fixture of tests/conftest.py
    bf, mean = synth.bitfield_from_grid_numpy(grid)
    o, d, img, poses = synth.ray_batch(4096, seed=1)
    scene = dict(grid=grid, bitfield=bf, mean=mean, rays_o=o, rays_d=d, img_ids=img, poses=poses, metadata=synth.metadata_for(poses.shape[0]))
    ot, dt, bft = T.scene_rays(scene)
    cr, _, nr, cntr = T._march(ref, ot, dt, bft, ot.shape[0] * 256)   # first call of the process: the reference's static pcg32 is at its seed
    counts, bases, crn = nr[:, 0].cpu().numpy(), nr[:, 1].cpu().numpy(), cr.cpu().numpy()
    rays = T.coord_rays(counts)
    coords = np.concatenate([crn[bases[i]:bases[i] + counts[i]] for i in rays])
    rgb, alpha = T.composite(ref, *T.composite_inputs(Port(), scene))
    np.savez_compressed(out_path, ns=counts, cnt=cntr.cpu().numpy(), rays=rays, coords=coords, rgb=rgb, alpha=alpha)
    print('wrote', out_path, os.path.getsize(out_path), 'bytes')


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else T.GOLDEN)
