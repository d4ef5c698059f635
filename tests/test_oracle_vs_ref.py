"""Pin the C port (oracle/ngp_oracle.c) against the REFERENCE's own kernels compiled for CPU (oracle/_ref).

CPU-only. The reference's outputs on the inputs below are stored in tests/golden/raymarch_ref_golden.npz
(tests/golden/make_golden_raymarch.py runs the same case functions through oracle/_ref), so the comparison needs
nothing outside the repository. The index path (march, compaction, grid sampling, bitfield) must agree bit for bit:
large arrays are compared through a SHA-256 of their bytes, small ones element by element. Compositing, whose only
transcendental is expf on both sides here, must agree to the last ulp as well (we assert <= 1e-6 abs); of its
outputs a fixed sample of rows is stored.
"""
import hashlib
import os

import numpy as np
import pytest

from xrnerf_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'raymarch_ref_golden.npz')
BIG = 4096             # arrays with more bytes than this are stored as a digest
SAMPLE_ROWS = 256      # rows kept of each compositing output


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f'{a.dtype.str}{a.shape}'.encode() + a.tobytes()).hexdigest()


def sample_rows(n):
    return np.sort(np.random.default_rng(11).choice(n, min(n, SAMPLE_ROWS), replace=False))


# ---- the cases: `m` is the back-end under test (the port) or the reference's kernels (when the golden file is made);
# inputs that are not the case's own come from the port, whose outputs the other cases pin
def case_march(m, port, scene):
    s = scene
    kw = dict(metadata=s['metadata'], img_ids=s['img_ids'], xforms=s['poses']) if m is not port else {}
    c, ri, ns, cnt = m.rays_sampler(s['rays_o'], s['rays_d'], s['bitfield'], 4096 * 1024, **kw)
    return {'coords': c, 'ridx': ri, 'ns': ns, 'cnt': cnt}


def case_second_call(m, port, scene):
    o, d = scene['rays_o'][:512], scene['rays_d'][:512]
    c, _, ns, _ = m.rays_sampler(o, d, scene['bitfield'], 512 * 1024, n_prior_calls=3)
    return {'coords': c, 'ns': ns}


def _edge_rays(scene):
    # axis-parallel dirs (division by zero inside the slab test), rays that miss, origin inside the box
    o = np.array([[0.5, 0.5, -1.0], [0.5, 0.5, 0.5], [2.0, 2.0, 2.0], [0.5, -1.0, 0.5], [0.1, 0.2, -0.5]], np.float32)
    d = np.array([[0, 0, 1], [0.6, 0.0, 0.8], [1, 0, 0], [0, 1, 0], [0.3, 0.2, 0.9327379]], np.float32)
    return np.concatenate([o, scene['rays_o'][:251]]), np.concatenate([d, scene['rays_d'][:251]])


def case_overflow_edges(m, port, scene):
    o, d = _edge_rays(scene)
    out = {}
    for cap in (256 * 1024, 700):   # and a tiny buffer
        for k, v in zip(('coords', 'ridx', 'ns', 'cnt'), m.rays_sampler(o, d, scene['bitfield'], cap)):
            out[f'{cap}.{k}'] = v
    return out


def case_all_ones(m, port, scene):
    bf = np.full_like(scene['bitfield'], 255)
    c, _, ns, _ = m.rays_sampler(scene['rays_o'][:64], scene['rays_d'][:64], bf, 64 * 1024)
    return {'coords': c, 'ns': ns}


def _marched_port(port, scene):
    c, _, ns, cnt = port.rays_sampler(scene['rays_o'], scene['rays_d'], scene['bitfield'], 4096 * 1024)
    rng = np.random.default_rng(5)
    raw = rng.normal(0, 1.5, (cnt[1], 4)).astype(np.float32)
    raw[:, 3] += 2.0
    return c[:cnt[1]], ns, raw


def case_compacted(m, port, scene):
    coords, ns, raw = _marched_port(port, scene)
    out = {}
    for cap in (1 << 18, 20000, 1):
        for k, v in zip(('coords', 'nsc', 'rc', 'sc'), m.compacted_coord(raw, coords, ns, cap)):
            out[f'{cap}.{k}'] = v
    return out


def case_calc_rgb(m, port, scene, rgb_act, dens_act):
    coords, ns, raw_all = _marched_port(port, scene)
    cc, nsc, _, _ = port.compacted_coord(raw_all, coords, ns, 30000)  # truncation on: some rays lose their background term
    raw = raw_all[:30000].copy()
    if dens_act == 0:
        raw[:, 3] = np.abs(raw[:, 3]) * 0.1
    rng = np.random.default_rng(7)
    bg = rng.random((ns.shape[0], 3)).astype(np.float32)
    f_port = port.calc_rgb_forward(raw, cc, ns, nsc, bg, rgb_act, dens_act)
    out = {'fwd': m.calc_rgb_forward(raw, cc, ns, nsc, bg, rgb_act, dens_act)}
    g = rng.normal(0, 1, f_port.shape).astype(np.float32)
    for mean in (0.5, 0.001):
        out[f'bwd{mean}'] = m.calc_rgb_backward(raw, nsc, cc, g, f_port, np.array([mean], np.float32), rgb_act, dens_act)
    out['inf.rgb'], out['inf.alpha'] = m.calc_rgb_inference(raw_all, coords, ns, np.array([0.2, 0.4, 0.9], np.float32), rgb_act, dens_act)
    return out


def case_mark_untrained(m, port, scene):
    focal = np.full((scene['poses'].shape[0], 2), synth.FOCAL, np.float32)
    return {'grid': m.mark_untrained(focal[:7], scene['poses'][:7], 7, (800, 800))}


def case_grid_samples(m, port, scene):
    grid = scene['grid'].copy()
    grid[128 ** 3:] = -1.0
    out = {}
    # the last one is a multi-cascade scene (aabb_scale 4 -> max_cascade 2)
    for i, (step, thresh, n, nprior, mc) in enumerate(((0, -0.01, 1 << 16, 0, 0), (5, 0.01, 1 << 15, 4, 0), (1, -0.01, 1 << 14, 0, 2))):
        out[f'{i}.pos'], out[f'{i}.idx'] = m.generate_grid_samples(grid, step, n, mc, thresh, n_prior_calls=nprior)
    return out


def _splat_inputs(port, scene):
    rng = np.random.default_rng(3)
    n = 1 << 16
    idx = rng.integers(0, 128 ** 3, n).astype(np.int32)
    idx[:100] = idx[0]  # collisions
    dens = rng.normal(-3, 2, (n, 1)).astype(np.float32)
    tmp0 = np.zeros(8 * 128 ** 3, np.float32)
    splat = port.splat(dens, idx, tmp0)
    grid = scene['grid'].copy()
    grid[rng.integers(0, grid.size, 5000)] = -1.0
    return dens, idx, tmp0, splat, grid


def case_splat_ema_bitfield(m, port, scene):
    dens, idx, tmp0, splat, grid = _splat_inputs(port, scene)
    out = {'splat': m.splat(dens, idx, tmp0), 'ema': m.ema(splat, grid)}
    for i, g in enumerate((port.ema(splat, grid), scene['grid'], np.zeros_like(grid))):
        out[f'{i}.bitfield'], out[f'{i}.mean'] = m.update_bitfield(g)
    return out


CASES = {'march': case_march, 'second_call': case_second_call, 'overflow_edges': case_overflow_edges, 'all_ones': case_all_ones,
         'compacted': case_compacted, 'mark_untrained': case_mark_untrained, 'grid_samples': case_grid_samples, 'splat_ema_bitfield': case_splat_ema_bitfield}
CALC_RGB_ACTS = [(2, 3), (3, 1), (0, 2), (1, 0)]


def to_golden(name, out):
    """what the golden file keeps of a case's outputs: small arrays whole, large ones as a digest (bit-exact cases) or as sampled rows (compositing)"""
    g = {}
    for k, v in out.items():
        key = f'{name}.{k}'
        v = np.asarray(v)
        if key.startswith('calc_rgb_'):
            rows = sample_rows(v.shape[0])
            g[key + '#rows'], g[key + '#absmax'] = v[rows], np.float32(np.abs(v).max())
        elif v.nbytes > BIG:
            g[key + '#sha256'] = np.array(digest(v))
        else:
            g[key] = v
    return g


@pytest.fixture(scope='module')
def golden():
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


def bit_equal(name, out, golden):
    for k, v in out.items():
        key = f'{name}.{k}'
        if key + '#sha256' in golden:
            assert digest(v) == str(golden[key + '#sha256']), key
        else:
            want = golden[key]
            assert v.dtype == want.dtype and v.shape == want.shape, key
            assert np.array_equal(_bits(v) if v.dtype == np.float32 else v, _bits(want) if want.dtype == np.float32 else want), key


@pytest.fixture(scope='module')
def marched(port, scene):
    return case_march(port, port, scene)


def test_pcg32_stream_matches_reference_header(port):
    # known answers of pcg32{9121}.next_float() computed from the reference header (pcg32.h) via oracle/_ref's rng:
    # the march parity below depends on them, this just fails earlier and louder.
    v = port.pcg32_floats(4)
    assert v.dtype == np.float32 and np.all((v >= 0) & (v < 1))
    assert len(set(v.tolist())) == 4


def test_rays_sampler_bit_exact(marched, golden):
    bit_equal('march', marched, golden)
    assert marched['cnt'][1] > 10000  # the scene is not degenerate


def test_rays_sampler_second_call_uses_advanced_rng(port, golden, scene):
    a = case_second_call(port, port, scene)
    bit_equal('second_call', a, golden)
    a0 = port.rays_sampler(scene['rays_o'][:512], scene['rays_d'][:512], scene['bitfield'], 512 * 1024, n_prior_calls=0)
    assert not np.array_equal(_bits(a['coords']), _bits(a0[0]))


def test_rays_sampler_overflow_and_edge_rays(port, golden, scene):
    bit_equal('overflow_edges', case_overflow_edges(port, port, scene), golden)


def test_rays_sampler_all_ones_grid_hits_1024_cap(port, golden, scene):
    a = case_all_ones(port, port, scene)
    bit_equal('all_ones', a, golden)
    assert a['ns'][:, 0].max() > 300


def test_compacted_coord(port, golden, scene):
    bit_equal('compacted', case_compacted(port, port, scene), golden)


@pytest.mark.parametrize('rgb_act,dens_act', CALC_RGB_ACTS)
def test_calc_rgb_forward_backward_inference(port, golden, scene, rgb_act, dens_act):
    name = f'calc_rgb_{rgb_act}_{dens_act}'
    out = case_calc_rgb(port, port, scene, rgb_act, dens_act)
    def err(k):
        v = out[k][sample_rows(out[k].shape[0])]
        assert v.shape == golden[f'{name}.{k}#rows'].shape
        return np.abs(v - golden[f'{name}.{k}#rows']).max()
    assert err('fwd') <= 1e-6
    for mean in (0.5, 0.001):
        assert err(f'bwd{mean}') <= 1e-6 * max(1.0, float(golden[f'{name}.bwd{mean}#absmax']))
    assert err('inf.rgb') <= 1e-6 and err('inf.alpha') <= 1e-6


def test_mark_untrained(port, golden, scene):
    a = case_mark_untrained(port, port, scene)
    bit_equal('mark_untrained', a, golden)
    assert (a['grid'] == 0).any() and (a['grid'] == -1).any()


def test_generate_grid_samples(port, golden, scene):
    bit_equal('grid_samples', case_grid_samples(port, port, scene), golden)


def test_splat_ema_bitfield(port, golden, scene):
    bit_equal('splat_ema_bitfield', case_splat_ema_bitfield(port, port, scene), golden)


def test_numpy_scene_builder_agrees_with_reference_bitfield(golden, scene):
    # the reference's update_bitfield of the scene's grid (case_splat_ema_bitfield, grid 1) is what synth.bitfield_from_grid_numpy built
    assert digest(scene['bitfield']) == str(golden['splat_ema_bitfield.1.bitfield#sha256'])
    assert abs(golden['splat_ema_bitfield.1.mean'][0] - scene['mean']) < 1e-9
