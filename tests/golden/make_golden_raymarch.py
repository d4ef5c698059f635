"""Generates tests/golden/raymarch_ref_golden.npz: the REFERENCE's own ngp_raymarch kernels compiled for CPU (oracle/_ref, built by
`make -C oracle ref` where the reference sources are present) run on the inputs of every case in tests/test_oracle_vs_ref.py.

    python tests/golden/make_golden_raymarch.py

The .npz is committed; the tests only read it.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
from oracle.oracle import Port, Ref, build, have_ref  # noqa: E402
from xrnerf_b200 import synth  # noqa: E402
import test_oracle_vs_ref as T  # noqa: E402


def main():
    build()
    assert have_ref(), 'oracle/_ref/libraymarch_ref.so is not built'
    port, ref = Port(), Ref(serial=True)
    grid = synth.lego_like_density_grid(0)       # the `scene` fixture of tests/conftest.py
    bf, mean = synth.bitfield_from_grid_numpy(grid)
    o, d, img, poses = synth.ray_batch(4096, seed=1)
    scene = dict(grid=grid, bitfield=bf, mean=mean, rays_o=o, rays_d=d, img_ids=img, poses=poses, metadata=synth.metadata_for(poses.shape[0]))
    out = {}
    for name, fn in T.CASES.items():
        out.update(T.to_golden(name, fn(ref, port, scene)))
    for ra, da in T.CALC_RGB_ACTS:
        out.update(T.to_golden(f'calc_rgb_{ra}_{da}', T.case_calc_rgb(ref, port, scene, ra, da)))
    np.savez_compressed(T.GOLDEN, **out)
    print('wrote', T.GOLDEN, 'with', len(out), 'arrays,', os.path.getsize(T.GOLDEN), 'bytes')


if __name__ == '__main__':
    main()
