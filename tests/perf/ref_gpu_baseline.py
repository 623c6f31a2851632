"""Reference-GPU baseline on the same B200 (BASELINE.md §2a): the reference's OWN CUDA kernels (oracle/_ref, built unmodified
except -std=c++17) driven by the reference's host loop (base_volume_renderer.py:79-123) with PyTorch decode, and the UNet as
plain PyTorch/cuDNN modules in the reference's default precision (fp32 storage, TF32 convs allowed, cudnn.benchmark) plus fp16
autocast.  Measurement tool only (not imported by the product)."""
import json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle', '_ref'))
import torch
import torch.nn.functional as F
from oracle import render_port as rp, unet_port as up
from bench import orbit_poses
import _raymarching as rmref, _shencoder as shref
dev = torch.device('cuda:0')
torch.backends.cudnn.benchmark = True


def ref_render(params, code_single, bf, ro, rd, max_steps=256):
    from tests.golden.make_golden_ref_kernels import reference_eval_loop
    return reference_eval_loop(rmref, shref, params, ro, rd, code_single, bf, max_steps=max_steps)


def time_render(V):
    g = torch.Generator().manual_seed(0)
    code = torch.randn(1, 3, 6, 128, 128, generator=g).clamp(-2, 2).to(dev)
    params = rp.make_decoder_params('P', 0, nonzero_dir=False)
    rands = [torch.rand(64 ** 3, 3, generator=g)]
    _, bf = rp.get_density(params, code.cpu(), rands, density_thresh=0.1)
    bf = torch.from_numpy(bf[0]).to(dev)
    poses = orbit_poses(251)[:V]
    intr = torch.tensor([131.25, 131.25, 64.0, 64.0]).expand(V, 4).contiguous()
    ro, rd = rp.get_cam_rays(poses, intr, 128, 128)
    ro, rd = ro.reshape(-1, 3).contiguous().to(dev), rd.reshape(-1, 3).contiguous().to(dev)
    ref_render(params, code[0], bf, ro, rd)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ws, dep, img = ref_render(params, code[0], bf, ro, rd)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    # ours on the same inputs
    from ssdnerf_b200 import renderer as R
    blob = R.pack_decoder_blob(params, R.DEC_P, device=dev)
    planes = R.pack_planes(code, R.DEC_P)
    for _ in range(2):
        out = R.render_fwd(R.DEC_P, planes, (128, 128), bf[None], blob, rays_o=ro[None], rays_d=rd[None])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = R.render_fwd(R.DEC_P, planes, (128, 128), bf[None], blob, rays_o=ro[None], rays_d=rd[None])
    e1.record(); torch.cuda.synchronize()
    ours = e0.elapsed_time(e1) * 1e-3
    err = float((out['image'][0] - img).abs().max())
    n = ro.shape[0]
    return dict(views=V, rays=n, ref_s=dt, ref_rays_per_s=n / dt, ours_s=ours, ours_rays_per_s=n / ours, speedup=dt / ours, max_abs_diff_image=err)


def time_unet(B, autocast):
    spec = up.unet_spec()
    sd = {k: v.to(dev) for k, v in up.random_state_dict(spec, seed=0).items()}
    x = torch.randn(B, 18, 128, 128, device=dev)
    t = torch.full((B,), 500, device=dev, dtype=torch.long)
    ctx = torch.autocast('cuda', dtype=torch.float16) if autocast else torch.autocast('cuda', enabled=False)
    with torch.no_grad(), ctx:
        for _ in range(3):
            up_forward_cuda(sd, spec, x, t)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            up_forward_cuda(sd, spec, x, t)
        e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    return dict(batch=B, autocast_fp16=autocast, ms_per_unet_eval=ms, triplanes_per_s=B / (ms * 1e-3 * 50))


def up_forward_cuda(sd, spec, x, t):
    # oracle functional UNet, tensors on the GPU; the time embedding helper builds its table on the CPU -> move it
    tt = t.float() * (1000.0 / 1000)
    half = spec['base'] // 2
    import math
    freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32, device=x.device) / half)
    args = tt[:, None] * freqs[None]
    e = torch.cat([torch.cos(args), torch.sin(args)], dim=-1)
    e = F.linear(e, sd['time_embedding.blocks.0.weight'], sd['time_embedding.blocks.0.bias'])
    emb = F.linear(F.silu(e), sd['time_embedding.blocks.2.weight'], sd['time_embedding.blocks.2.bias'])
    h, hs = x, []
    for layers in spec['in_blocks']:
        h = up._run_layers(sd, spec, layers, h, emb); hs.append(h)
    h = up._run_layers(sd, spec, spec['mid'], h, emb)
    for layers in spec['out_blocks']:
        h = up._run_layers(sd, spec, layers, torch.cat([h, hs.pop()], dim=1), emb)
    h = F.silu(F.group_norm(h, 32, sd['out.gn.weight'], sd['out.gn.bias'], eps=1e-5))
    return F.conv2d(h, sd['out.conv.weight'], sd['out.conv.bias'], padding=1)


if __name__ == '__main__':
    res = dict(render=[time_render(V) for V in (1, 8, 32, 128, 251)], unet=[time_unet(16, False), time_unet(16, True)])
    print(json.dumps(res, indent=1))
