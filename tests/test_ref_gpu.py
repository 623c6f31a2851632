"""Parity against the REFERENCE'S OWN CUDA kernels (lib/ops/raymarching, lib/ops/shencoder compiled unmodified except -std=c++17),
through their outputs on these same seeded inputs, stored in tests/golden/reference_kernels_v1.npz by
tests/golden/make_golden_ref_kernels.py on a B200.  Integer / index outputs and the marcher's floats are compared bit-exactly (SHA-256 of
the whole array, and a sample of rows for the message); compositor floats to 1e-6 (both use MUFU.EX2 based __expf), element by element
except the per-sample gradients of the training compositor, which are compared on a sample of rows and on their per-channel sums."""
import numpy as np
import pytest
import torch

from oracle import render_port as rp
from tests.golden import make_golden_ref_kernels as G

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def gold():
    return dict(np.load(G.GOLDEN))


def _inputs(gold, scenario, *arrays):
    assert np.array_equal(G.sha256(*arrays), gold[scenario + '.inputs']), \
        f'{scenario}: the inputs differ from those the stored reference outputs were computed on'


def _check(gold, key, t, rtol=None, atol=None):
    """bit-exact when no tolerance is given, else |a - ref| <= atol + rtol * |ref| on every element stored (and, for a stored sample of
    rows, its consequence on the per-channel sums)"""
    a = G.host(t)
    assert a.shape == tuple(gold[key + '.shape']), f'{key}: shape {a.shape} vs {tuple(gold[key + ".shape"])}'
    if key + '.value' in gold:
        np.testing.assert_allclose(a, gold[key + '.value'], rtol=rtol, atol=atol, err_msg=key)
        return
    ref = gold[key + '.sample']
    got = a[G.sample_index(len(a), len(ref))]
    if rtol is None:
        bits = f'u{a.itemsize}'
        np.testing.assert_array_equal(got.view(bits), ref.view(bits), err_msg=key)
        assert np.array_equal(G.sha256(a), gold[key + '.sha256']), f'{key}: the sampled rows agree, others differ'
    else:
        np.testing.assert_allclose(got, ref, rtol=rtol, atol=atol, err_msg=key)
        s, s_abs = gold[key + '.sum']
        assert np.all(np.abs(a.sum(0, dtype=np.float64) - s) <= len(a) * atol + rtol * s_abs), key


def test_utils_bit_exact(cuda, gold):
    from ssdnerf_b200 import raymarching as rm
    ro, rd = G.cam_rays(cuda)
    coords, grid = G.utils_inputs(cuda)
    _inputs(gold, 'utils', ro, rd, coords, grid)
    n, f = rm.near_far_from_aabb(ro, rd, G.aabb(cuda), 0.2)
    _check(gold, 'utils.near', n)
    _check(gold, 'utils.far', f)
    _check(gold, 'utils.morton', rm.morton3D(coords))
    for name, gq in (('f32', grid), ('f16', grid.half())):
        _check(gold, f'utils.packbits_{name}', rm.packbits(gq, 0.41))


@pytest.mark.parametrize('dt_gamma', G.DT_GAMMAS)
def test_march_and_composite_bit_exact(cuda, gold, dt_gamma):
    from ssdnerf_b200 import raymarching as rm
    i = G.DT_GAMMAS.index(dt_gamma)
    ro, rd = G.cam_rays(cuda)
    N = ro.shape[0]
    nears, fars = rm.near_far_from_aabb(ro, rd, G.aabb(cuda), 0.2)
    bf = torch.from_numpy(rp.sphere_bitfield()).to(cuda)
    sig, rgb = G.composite_inputs(G.march_steps(N))
    _inputs(gold, 'march', ro, rd, bf, sig, rgb)
    alive = torch.arange(N, dtype=torch.int32, device=cuda)
    rays_t = nears.clone()
    outs = rm.march_rays(N, 3, alive, rays_t, ro, rd, 1.0, bf, 1, 64, nears, fars, align=128, dt_gamma=dt_gamma, max_steps=256)
    for name, t in zip(('xyzs', 'dirs', 'deltas'), outs):
        _check(gold, f'march{i}.{name}', t)
    st = [alive, rays_t, torch.zeros(N, device=cuda), torch.zeros(N, device=cuda), torch.zeros(N, 3, device=cuda)]
    rm.composite_rays(N, 3, st[0], st[1], sig.to(cuda), rgb.to(cuda), outs[2], st[2], st[3], st[4], 1e-4)
    _check(gold, f'march{i}.alive', st[0])
    _check(gold, f'march{i}.rays_t', st[1])
    for name, t in zip(('weights_sum', 'depth', 'image'), st[2:]):
        _check(gold, f'march{i}.{name}', t, rtol=1e-6, atol=1e-7)


def test_march_train_and_composite_train(cuda, gold):
    from ssdnerf_b200 import raymarching as rm
    ro, rd = G.cam_rays(cuda, res=32)
    N = ro.shape[0]
    nears, fars = rm.near_far_from_aabb(ro, rd, G.aabb(cuda), 0.2)
    bf = torch.from_numpy(rp.sphere_bitfield()).to(cuda)
    g = torch.Generator().manual_seed(2)
    noises = torch.rand(N, generator=g)
    xyz, dirs, deltas, rays = rm.march_rays_train(ro, rd, 1.0, bf, 1, 64, nears, fars, perturb=True, force_all_rays=True,
                                                  dt_gamma=0.0, max_steps=256, noises=noises.to(cuda))
    m = xyz.shape[0]
    r = G.host(rays)
    _check(gold, 'train.rays', r[np.argsort(r[:, 0], kind='stable')][:, [0, 2]])
    _check(gold, 'train.count', np.array([m], np.int64))
    five = torch.from_numpy(G.ray_major(rays, every=5)).to(cuda)
    _check(gold, 'train.xyzs', xyz[five])
    _check(gold, 'train.deltas', deltas[five])
    # compositing forward / backward of the same seeded per-sample values, drawn in ray-major order
    perm = torch.from_numpy(G.ray_major(rays)).to(cuda)
    sig_c, rgb_c = torch.rand(m, generator=g) * 20, torch.rand(m, 3, generator=g)
    gws, gimg = torch.rand(N, generator=g), torch.rand(N, 3, generator=g)
    _inputs(gold, 'train', ro, rd, bf, noises, sig_c, rgb_c, gws, gimg)
    sig, rgb = torch.empty(m, device=cuda), torch.empty(m, 3, device=cuda)
    sig[perm], rgb[perm] = sig_c.to(cuda), rgb_c.to(cuda)
    sig_g, rgb_g = sig.requires_grad_(True), rgb.requires_grad_(True)
    ws, dep, img = rm.composite_rays_train(sig_g, rgb_g, deltas, rays, 1e-4)
    _check(gold, 'train.weights_sum', ws, rtol=1e-6, atol=1e-7)
    _check(gold, 'train.image', img, rtol=1e-6, atol=1e-7)
    torch.autograd.backward([ws, img], [gws.to(cuda), gimg.to(cuda)])
    _check(gold, 'train.grad_sigmas', sig_g.grad[perm], rtol=1e-5, atol=1e-6)
    _check(gold, 'train.grad_rgbs', rgb_g.grad[perm], rtol=1e-6, atol=1e-7)


def test_sh_encode_bit_exact(cuda, gold):
    from ssdnerf_b200.shencoder import sh_encode
    d = G.sh_inputs(cuda)
    _inputs(gold, 'sh', d)
    _check(gold, 'sh.out', sh_encode(d, 4, False))


def test_fused_renderer_vs_reference_pipeline(cuda, gold):
    """whole eval renderer: reference kernels + PyTorch decode (fp32, TF32 off) vs the fused kernel, variant P"""
    from ssdnerf_b200 import renderer as R
    code, params = G.render_inputs(cuda)
    ro, rd = G.cam_rays(cuda)
    bf = torch.from_numpy(rp.sphere_bitfield()).to(cuda)
    _inputs(gold, 'render', code, ro, rd, bf, *[params[k] for k in sorted(params)])
    out = R.render_fwd(R.DEC_P, R.pack_planes(code, R.DEC_P), (128, 128), bf[None], R.pack_decoder_blob(params, R.DEC_P, device=cuda),
                       rays_o=ro[None], rays_d=rd[None], max_steps=256)
    _check(gold, 'render.weights_sum', out['weights_sum'][0], rtol=2e-4, atol=2e-5)
    _check(gold, 'render.image', out['image'][0], rtol=2e-4, atol=2e-5)
    _check(gold, 'render.depth', out['depth'][0], rtol=2e-4, atol=1e-4)
