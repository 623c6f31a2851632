"""Outputs of the reference's OWN CUDA kernels (lib/ops/raymarching, lib/ops/shencoder, compiled unmodified except -std=c++17 into
oracle/_ref by oracle/build_ref.sh) on the seeded inputs of tests/test_ref_gpu.py, and of the reference's eval loop
(base_volume_renderer.py:79-123) driven by them  ->  tests/golden/reference_kernels_v1.npz.  Run on a B200 once oracle/_ref is built:

    python tests/golden/make_golden_ref_kernels.py [OUT.npz]

An output the test compares bit-exactly is stored as the SHA-256 of its bytes plus an evenly spaced sample of its rows (for the failure
message).  An output compared to a tolerance is stored whole, except the per-sample gradients of the training compositor, which are stored
as an evenly spaced sample of their rows plus their per-channel sums and absolute sums.  Each scenario also stores the SHA-256 of its
inputs, so that a change of the inputs is reported as such."""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import render_port as rp  # noqa: E402
from tests.common import spiral_poses  # noqa: E402

GOLDEN = os.path.join(HERE, 'reference_kernels_v1.npz')
DT_GAMMAS = (0.0, 0.0078125)


def host(t):
    return t.detach().cpu().contiguous().numpy() if torch.is_tensor(t) else np.ascontiguousarray(t)


def sha256(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(host(a).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def sample_index(n, k):
    """min(n, k) evenly spaced indices into n rows"""
    return np.unique(np.linspace(0, n - 1, min(n, k)).round().astype(np.int64))


def record(out, key, t, exact=False, rows=None):
    """exact: SHA-256 + 256 sample rows; else the whole array, or with `rows`: that many sample rows + per-channel (abs) sums"""
    a = host(t)
    out[key + '.shape'] = np.array(a.shape, np.int64)
    if exact:
        out[key + '.sha256'] = sha256(a)
        out[key + '.sample'] = a[sample_index(len(a), 256)]
    elif rows is None:
        out[key + '.value'] = a
    else:
        out[key + '.sample'] = a[sample_index(len(a), rows)]
        out[key + '.sum'] = np.stack([a.sum(0, dtype=np.float64), np.abs(a).sum(0, dtype=np.float64)])


def ray_major(rays, every=1):
    """indices of the samples of a march_rays_train output, ray by ray in ray-index order, for every `every`-th ray; the reference
    lays the rays out in atomicAdd arrival order, so its outputs are compared in this order"""
    r = host(rays)
    r = r[np.argsort(r[:, 0], kind='stable')][::every]
    return np.concatenate([np.arange(o, o + c, dtype=np.int64) for _, o, c in r])


def aabb(dev):
    return torch.tensor([-1., -1, -1, 1, 1, 1], device=dev)


def cam_rays(dev, res=64, V=2):
    poses = torch.from_numpy(spiral_poses(V))
    intr = torch.tensor([res * 131.25 / 128, res * 131.25 / 128, res / 2, res / 2]).expand(V, 4).contiguous()
    ro, rd = rp.get_cam_rays(poses, intr, res, res)
    return ro.reshape(-1, 3).contiguous().to(dev), rd.reshape(-1, 3).contiguous().to(dev)


def utils_inputs(dev):
    g = torch.Generator().manual_seed(0)
    coords = torch.randint(0, 128, (50000, 3), generator=g, dtype=torch.int32).to(dev)
    grid = torch.rand(2, 64 ** 3, generator=g).to(dev)
    return coords, grid


def composite_inputs(M):
    g = torch.Generator().manual_seed(1)
    return torch.rand(M, generator=g) * 30, torch.rand(M, 3, generator=g)


def march_steps(N, n_step=3, align=128):
    M = N * n_step
    return M + align - M % align


def render_inputs(dev):
    g = torch.Generator().manual_seed(4)
    code = torch.randn(1, 3, 6, 128, 128, generator=g).clamp(-2, 2).to(dev)
    return code, rp.make_decoder_params('P', 5)


def ref_utils(rmref, dev, out):
    ro, rd = cam_rays(dev)
    N = ro.shape[0]
    n, f = torch.empty(N, device=dev), torch.empty(N, device=dev)
    rmref.near_far_from_aabb(ro, rd, aabb(dev), N, 0.2, n, f)
    coords, grid = utils_inputs(dev)
    idx = torch.empty(50000, dtype=torch.int32, device=dev)
    rmref.morton3D(coords, 50000, idx)
    out['utils.inputs'] = sha256(ro, rd, coords, grid)
    record(out, 'utils.near', n, True)
    record(out, 'utils.far', f, True)
    record(out, 'utils.morton', idx, True)
    for name, gq in (('f32', grid), ('f16', grid.half())):
        bits = torch.empty(2 * 64 ** 3 // 8, dtype=torch.uint8, device=dev)
        rmref.packbits(gq.contiguous(), 2 * 64 ** 3 // 8, 0.41, bits)
        record(out, f'utils.packbits_{name}', bits, True)


def ref_march_and_composite(rmref, dev, out):
    ro, rd = cam_rays(dev)
    N = ro.shape[0]
    nears, fars = torch.empty(N, device=dev), torch.empty(N, device=dev)
    rmref.near_far_from_aabb(ro, rd, aabb(dev), N, 0.2, nears, fars)
    bf = torch.from_numpy(rp.sphere_bitfield()).to(dev)
    n_step, M = 3, march_steps(N)
    sig, rgb = composite_inputs(M)
    out['march.inputs'] = sha256(ro, rd, bf, sig, rgb)
    sig, rgb = sig.to(dev), rgb.to(dev)
    for i, dt_gamma in enumerate(DT_GAMMAS):
        alive = torch.arange(N, dtype=torch.int32, device=dev)
        rays_t = nears.clone()
        outs = [torch.zeros(M, 3, device=dev), torch.zeros(M, 3, device=dev), torch.zeros(M, 2, device=dev)]
        rmref.march_rays(N, n_step, alive, rays_t, ro, rd, 1.0, dt_gamma, 256, 1, 64, bf, nears, fars, *outs, torch.zeros(N, device=dev))
        for name, t in zip(('xyzs', 'dirs', 'deltas'), outs):
            record(out, f'march{i}.{name}', t, True)
        st = [alive, rays_t, torch.zeros(N, device=dev), torch.zeros(N, device=dev), torch.zeros(N, 3, device=dev)]
        rmref.composite_rays(N, n_step, 1e-4, st[0], st[1], sig, rgb, outs[2], st[2], st[3], st[4])
        record(out, f'march{i}.alive', st[0], True)
        record(out, f'march{i}.rays_t', st[1], True)
        for name, t in zip(('weights_sum', 'depth', 'image'), st[2:]):
            record(out, f'march{i}.{name}', t)


def ref_march_train_and_composite_train(rmref, dev, out):
    ro, rd = cam_rays(dev, res=32)
    N = ro.shape[0]
    nears, fars = torch.empty(N, device=dev), torch.empty(N, device=dev)
    rmref.near_far_from_aabb(ro, rd, aabb(dev), N, 0.2, nears, fars)
    bf = torch.from_numpy(rp.sphere_bitfield()).to(dev)
    g = torch.Generator().manual_seed(2)
    noises = torch.rand(N, generator=g)
    M = N * 256
    xyz, dirs, deltas = torch.zeros(M, 3, device=dev), torch.zeros(M, 3, device=dev), torch.zeros(M, 2, device=dev)
    rays, cnt = torch.empty(N, 3, dtype=torch.int32, device=dev), torch.zeros(2, dtype=torch.int32, device=dev)
    rmref.march_rays_train(ro, rd, bf, 1.0, 0.0, 256, N, 1, 64, M, nears, fars, xyz, dirs, deltas, rays, cnt, noises.to(dev))
    m = int(cnt[0])
    r = host(rays)
    record(out, 'train.rays', r[np.argsort(r[:, 0], kind='stable')][:, [0, 2]], True)
    record(out, 'train.count', np.array([m], np.int64), True)
    five = torch.from_numpy(ray_major(rays, every=5)).to(dev)
    record(out, 'train.xyzs', xyz[five], True)
    record(out, 'train.deltas', deltas[five], True)
    # compositing forward / backward of the same seeded per-sample values, drawn in ray-major order
    perm = torch.from_numpy(ray_major(rays)).to(dev)
    sig_c, rgb_c = torch.rand(m, generator=g) * 20, torch.rand(m, 3, generator=g)
    gws, gimg = torch.rand(N, generator=g), torch.rand(N, 3, generator=g)
    out['train.inputs'] = sha256(ro, rd, bf, noises, sig_c, rgb_c, gws, gimg)
    sig, rgb = torch.empty(m, device=dev), torch.empty(m, 3, device=dev)
    sig[perm], rgb[perm] = sig_c.to(dev), rgb_c.to(dev)
    deltas = deltas[:m].contiguous()
    ws, dep, img = torch.empty(N, device=dev), torch.empty(N, device=dev), torch.empty(N, 3, device=dev)
    rmref.composite_rays_train_forward(sig, rgb, deltas, rays, m, N, 1e-4, ws, dep, img)
    record(out, 'train.weights_sum', ws)
    record(out, 'train.image', img)
    gs, gc = torch.zeros(m, device=dev), torch.zeros(m, 3, device=dev)
    rmref.composite_rays_train_backward(gws.to(dev), gimg.to(dev), sig, rgb, deltas, rays, ws, img, m, N, 1e-4, gs, gc)
    record(out, 'train.grad_sigmas', gs[perm], rows=2048)
    record(out, 'train.grad_rgbs', gc[perm], rows=2048)


def sh_inputs(dev):
    g = torch.Generator().manual_seed(3)
    return torch.nn.functional.normalize(torch.randn(10000, 3, generator=g), dim=-1).to(dev)


def ref_sh_encode(shref, dev, out):
    d = sh_inputs(dev)
    sh, dy = torch.empty(10000, 16, device=dev), torch.empty(10000, 48, device=dev)
    shref.sh_encode_forward(d, sh, 10000, 3, 4, True, dy)
    out['sh.inputs'] = sha256(d)
    record(out, 'sh.out', sh, True)


def reference_eval_loop(rmref, shref, params, ro, rd, code_single, bf, max_steps=256, T_thresh=1e-4):
    """the reference's eval branch (base_volume_renderer.py:79-123) driven with the reference's own kernels + torch decode"""
    dev = ro.device
    N = ro.shape[0]
    nears, fars = torch.empty(N, device=dev), torch.empty(N, device=dev)
    rmref.near_far_from_aabb(ro, rd, aabb(dev), N, 0.2, nears, fars)
    ws, dep, img = torch.zeros(N, device=dev), torch.zeros(N, device=dev), torch.zeros(N, 3, device=dev)
    alive = torch.arange(N, dtype=torch.int32, device=dev)
    rays_t = nears.clone()
    p = {k: v.to(dev) for k, v in params.items()}
    step = 0
    F = torch.nn.functional
    while step < max_steps:
        n_alive = alive.shape[0]
        if n_alive == 0:
            break
        n_step = min(max(N // n_alive, 1), 8)
        M = n_alive * n_step
        M += 128 - M % 128
        xyzs, dirs, deltas = torch.zeros(M, 3, device=dev), torch.zeros(M, 3, device=dev), torch.zeros(M, 2, device=dev)
        rmref.march_rays(n_alive, n_step, alive, rays_t, ro, rd, 1.0, 0.0, max_steps, 1, 64, bf, nears, fars, xyzs, dirs, deltas,
                         torch.zeros(n_alive, device=dev))
        pc = F.grid_sample(code_single, rp.xyz_transform(xyzs), mode='bilinear', padding_mode='border', align_corners=False).squeeze(-2)
        pc = pc.permute(2, 1, 0).reshape(M, -1)
        base_x = F.linear(pc, p['base_net.0.weight'], p['base_net.0.bias'])
        sig = torch.exp(F.linear(F.silu(base_x), p['density_net.0.weight'], p['density_net.0.bias'])).squeeze(-1)
        sh = torch.empty(M, 16, device=dev)
        shref.sh_encode_forward(dirs.contiguous(), sh, M, 3, 4, False, torch.empty(1, device=dev))
        rgb = torch.sigmoid(F.linear(F.silu(base_x + F.linear(sh, p['dir_net.0.weight'], p['dir_net.0.bias'])),
                                     p['color_net.0.weight'], p['color_net.0.bias'])) * 1.002 - 0.001
        rmref.composite_rays(n_alive, n_step, T_thresh, alive, rays_t, sig.contiguous(), rgb.contiguous(), deltas, ws, dep, img)
        alive = alive[alive >= 0]
        step += n_step
    return ws, dep, img


def ref_render(rmref, shref, dev, out):
    """whole eval renderer: reference kernels + PyTorch decode (fp32, TF32 off), variant P"""
    torch.backends.cuda.matmul.allow_tf32 = False
    code, params = render_inputs(dev)
    ro, rd = cam_rays(dev)
    bf = torch.from_numpy(rp.sphere_bitfield()).to(dev)
    out['render.inputs'] = sha256(code, ro, rd, bf, *[params[k] for k in sorted(params)])
    ws, dep, img = reference_eval_loop(rmref, shref, params, ro, rd, code[0], bf)
    for name, t in (('weights_sum', ws), ('image', img), ('depth', dep)):
        record(out, f'render.{name}', t)


def main(path):
    sys.path.insert(0, os.path.join(ROOT, 'oracle', '_ref'))
    import _raymarching
    import _shencoder
    dev = torch.device('cuda:0')
    out = {}
    ref_utils(_raymarching, dev, out)
    ref_march_and_composite(_raymarching, dev, out)
    ref_march_train_and_composite_train(_raymarching, dev, out)
    ref_sh_encode(_shencoder, dev, out)
    ref_render(_raymarching, _shencoder, dev, out)
    np.savez_compressed(path, **out)
    print(torch.cuda.get_device_name(dev), len(out), 'arrays,', os.path.getsize(path), 'bytes ->', path)


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else GOLDEN)
