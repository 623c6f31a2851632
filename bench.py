#!/usr/bin/env python
"""bench.py -- SSDNeRF hot-path benchmark (contract: see the task brief; numbers explained in DESIGN.md §6).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a kernels
    python bench.py --impl reference --steps K --warmup W    # reference arithmetic on the host cores (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR  # + the last timed step's outputs as DIR/<name>.npy

Every GPU measurement times K steps (calls); the `cpu_baseline` field is a fixed, bounded CPU sample (`--impl reference` times K of them).

Workload (BASELINE.json configs[1]): `ssdnerf_cars_uncond`, batch 16 scenes per GPU, one STEP =
    50-step DDIM sample of a (3,6,128,128) triplane batch  ->  8-iteration occupancy-grid build  ->
    251-view 128x128 render of every scene (4.1 M rays per scene),
model built from the REFERENCE's own config (tests/golden/reference_configs.json = configs/paper_cfgs/ssdnerf_cars_uncond.py resolved),
random-init weights (UNet convs re-drawn N(0, 0.02) because the reference zero-inits half of them), synthetic noise and a synthetic
251-pose camera orbit.  Scenes are independent, so N GPUs run N independent batches (weak scaling); the one exchange of the reference's
eval path -- the per-batch all-gather of lib/apis/test.py:41-53 -- runs on NCCL inside `e2e` at N > 1 (8-bit images, side stream,
overlapped with the next batch's DDIM).

`value`   = rays/s of the render stage, inputs resident in HBM (CUDA events on the launching stream, max over ranks)
`triplanes_per_sec` = batch / DDIM-stage time, same measurement
`e2e`     = the same step through the public plugin API (`DiffusionNeRF.val_step`) with PINNED HOST inputs, the device->host read of
            the rendered images and (N > 1) the NCCL all-gather inside the timed region; e2e.value = rays / whole-step time.
`render_variant_S` = north_star's synthetic workload (random-init 3x32x128x128 triplanes, class-default decoder, 251 views), every rank
`strong_scaling`   = ONE scene x 251 views sharded by view over the N ranks (broadcast planes + bitfield, gather the images)
`guided`           = config-4 shape (8 scenes, one 128x128 conditioning view): guided evaluations/s (UNet fwd + render loss fwd/bwd +
                     UNet input-gradient pass), rank 0
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU = 16
NUM_VIEWS = 251
IMG = 128
DDIM_STEPS = 50
METRIC = 'rays/sec (128^2 render) & DDIM triplanes/sec'
UNET_FLOP_PER_SAMPLE_STEP = 217.96e9     # SURVEY.md §8d / Appendix B
RAY_GATHER_BYTES_PER_SAMPLE = 288        # 3 planes x 4 taps x 6 ch x fp32 (SURVEY.md §8d)
RAY_IO_BYTES = 20                        # image[3] + depth + weights_sum per ray
DUMP_BYTES = 60_000_000                  # --dump-outputs writes at most this much array data (64 MB with the .npy headers)


def orbit_poses(num, radius=2.6):
    """synthetic stand-in for demo/camera_spiral_cars (251 poses at radius 1.3 x 2): look-at cameras on a sphere"""
    poses = []
    for i in range(num):
        phi = 2 * np.pi * i / num + 0.3
        theta = np.pi / 2 - 0.45 * np.sin(1.7 * phi)
        pos = radius * np.array([np.sin(theta) * np.cos(phi), np.sin(theta) * np.sin(phi), np.cos(theta)])
        fwd = -pos / np.linalg.norm(pos)
        right = np.cross(fwd, np.array([0.0, 0.0, 1.0])); right /= np.linalg.norm(right)
        down = np.cross(fwd, right)
        c2w = np.eye(4)
        c2w[:3, 0], c2w[:3, 1], c2w[:3, 2], c2w[:3, 3] = right, down, fwd, pos
        poses.append(c2w)
    return torch.from_numpy(np.stack(poses).astype(np.float32))


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], tf_burst=d['bf16_tflops'], tf_sustained=d.get('bf16_tflops_sustained', d['bf16_tflops']), src='measured')
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src='fallback')


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons while the timed region runs"""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.proc, self.lines, self.index = None, [], index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[2:6]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def dump_outputs(out_dir, arrays):
    """`arrays` as DIR/<name>.npy in float32.  The budget of DUMP_BYTES is shared out smallest array first; an array larger than its
    share is written as a sample of that many of its flattened elements, drawn with a fixed seed, so that two runs with the same
    arguments write the same elements."""
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES // 4
    for i, (name, t) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].numel())):
        share = left // (len(arrays) - i)
        a = t.detach()
        if a.numel() > share:
            idx = torch.randint(0, a.numel(), (share,), generator=torch.Generator().manual_seed(0)).sort().values
            a = a.reshape(-1)[idx.to(a.device)]
        left -= a.numel()
        np.save(os.path.join(out_dir, name + '.npy'), a.float().cpu().numpy())


# ----------------------------------------------------------------------------------------------------------- this repo
def reference_config(rel):
    """a config of the reference, resolved by tests/golden/make_config_fixtures.py (the GPU box has no /root/reference)"""
    return json.load(open(os.path.join(ROOT, 'tests', 'golden', 'reference_configs.json')))[rel]


def build_model(dev, seed=0, rel='configs/paper_cfgs/ssdnerf_cars_uncond.py', test_cfg_update=None):
    import ssdnerf_b200 as S
    cfg = reference_config(rel)
    test_cfg = dict(cfg['test_cfg'])
    test_cfg.update(test_cfg_update or {})
    torch.manual_seed(seed)
    model = S.build_model(cfg['model'], train_cfg=cfg['train_cfg'], test_cfg=test_cfg)
    g = torch.Generator().manual_seed(seed)
    for mod in (model.diffusion_ema.denoising, model.diffusion.denoising):
        for name, p in mod.named_parameters():
            if p.dim() > 1:
                p.data.copy_(torch.randn(p.shape, generator=g) * 0.02)     # non-degenerate UNet (SURVEY.md §8d config 2)
    return model.to(dev).eval(), cfg


def measured_traffic(kernel, rays):
    """DRAM bytes per launch of `kernel` from a committed `ncu --set full` capture of this bench command (profiles/r02_render_traffic.json,
    written by scripts/ncu_traffic.py from the .ncu-rep next to it); scaled by ray count when the capture used fewer views.  None when no
    capture of the current kernel is committed -- never a hard-coded constant."""
    path = os.path.join(ROOT, 'profiles', 'r02_render_traffic.json')
    if not os.path.exists(path):
        return None, None
    d = json.load(open(path)).get(kernel)
    if not d:
        return None, None
    return d['dram_bytes_per_launch'] * (rays / d['rays_per_launch']), f"profiles/r02_render_traffic.json ({d['source']})"


def run_ours(args):
    import ctypes
    import ssdnerf_b200 as S
    from ssdnerf_b200 import _lib as N
    from ssdnerf_b200 import density as Dm
    from ssdnerf_b200 import renderer as R
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', 0)); world = int(os.environ.get('WORLD_SIZE', 1)); local = int(os.environ.get('LOCAL_RANK', 0))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device; the hot path has no CPU fallback')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    model, cfg = build_model(dev, seed=0)
    diffusion, decoder = model.diffusion_ema, model.decoder_ema
    B, V = args.batch, args.views
    g = torch.Generator().manual_seed(1234 + rank)
    noise_host = torch.randn(B, *model.code_size, generator=g).pin_memory()
    poses_host = orbit_poses(V)[None].repeat(B, 1, 1, 1).contiguous().pin_memory()
    intr_host = torch.tensor([131.25, 131.25, 64.0, 64.0]).expand(B, V, 4).contiguous().pin_memory()
    rays = B * V * IMG * IMG
    L = N.lib()
    L.ssdnerf_launch_count.restype = ctypes.c_ulonglong

    noise, poses, intr = noise_host.to(dev), poses_host.to(dev), intr_host.to(dev)
    stream = torch.cuda.current_stream(dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, warmup):
        """`steps` calls of fn between CUDA events on the launching stream, barrier + synchronize on both sides -> ms per call"""
        for _ in range(warmup):
            fn()
        barrier()
        t0, t1 = ev(), ev()
        t0.record(stream)
        for _ in range(steps):
            fn()
        t1.record(stream)
        barrier()
        return t0.elapsed_time(t1) / steps

    def resident_step(rec=None):
        """one step with inputs already in HBM; stage boundaries marked with CUDA events on the launching stream -> what the step
        hands its caller"""
        e = [ev() for _ in range(4)]
        e[0].record(stream)
        code = model.code_diff_pr_inv(diffusion(model.code_diff_pr(noise), return_loss=False)).contiguous()
        e[1].record(stream)
        grid, bitfield = model.get_density(decoder, code, cfg=model.test_cfg)
        e[2].record(stream)
        img, depth = model.render(decoder, code, bitfield, IMG, IMG, intr, poses, cfg=model.test_cfg)
        e[3].record(stream)
        if rec is not None:
            rec.append(e)
        return dict(triplanes=code, density_grid=grid, density_bitfield=bitfield, image=img, depth=depth)

    # ---- end-to-end through the plugin API with host buffers (+ the eval-side NCCL all-gather of 8-bit images when N > 1)
    out_hosts = [torch.empty(B, V, 3, IMG, IMG, dtype=torch.float32).pin_memory() for _ in range(2)]
    out_host = out_hosts[0]
    copy_stream = torch.cuda.Stream(device=dev)         # D2H of batch i runs under the DDIM of batch i + 1 (double-buffered pinned memory)
    copy_done = [None, None]
    side = torch.cuda.Stream(device=dev) if world > 1 else None
    u8_bufs = [torch.empty(B * V, 3, IMG, IMG, dtype=torch.uint8, device=dev) for _ in range(2)] if world > 1 else None
    gathered = [torch.empty(world * B * V, 3, IMG, IMG, dtype=torch.uint8, device=dev) for _ in range(2)] if world > 1 else None
    pending = [None, None]
    e2e_state = dict(i=0)

    def e2e_step():
        """public API with host buffers: H2D inputs, val_step, D2H of the rendered images (lib/apis/test.py:27-53 data flow); at N > 1 the
        batch's images are quantised to 8 bits and all-gathered over NCCL on a side stream, overlapping the next batch's DDIM"""
        data = dict(scene_id=list(range(B)), scene_name=[str(i) for i in range(B)], noise=noise_host.to(dev, non_blocking=True),
                    test_poses=poses_host.to(dev, non_blocking=True), test_intrinsics=intr_host.to(dev, non_blocking=True))
        out = model.val_step(data)
        k = e2e_state['i'] & 1
        e2e_state['i'] += 1
        if world > 1:
            if pending[k] is not None:
                pending[k].wait()                      # the gather that last used this buffer pair
            u8_bufs[k].copy_((out['pred_imgs'].reshape(B * V, 3, IMG, IMG) * 255.0 + 0.5).to(torch.uint8))
            side.wait_stream(stream)
            with torch.cuda.stream(side):
                pending[k] = dist.all_gather_into_tensor(gathered[k], u8_bufs[k], async_op=True)
        if copy_done[k] is not None:
            copy_done[k].synchronize()                  # the host buffer is free again (its copy was issued two steps ago)
        copy_stream.wait_stream(stream)
        with torch.cuda.stream(copy_stream):
            out_hosts[k].copy_(out['pred_imgs'], non_blocking=True)
            out['pred_imgs'].record_stream(copy_stream)
            copy_done[k] = torch.cuda.Event()
            copy_done[k].record(copy_stream)
        return out

    def e2e_drain():
        for k in range(2):
            if pending[k] is not None:
                pending[k].wait()
                pending[k] = None
        if side is not None:
            stream.wait_stream(side)
        stream.wait_stream(copy_stream)                 # every device->host copy has landed before the closing event

    # ---- resident (kernel-side) measurement; warm-up and timed steps alike keep the previous step's outputs alive until the next returns
    for _ in range(args.warmup):
        last = resident_step()
    barrier()
    launches0 = L.ssdnerf_launch_count()
    clocks = ClockSampler(local); clocks.start()
    rec = []
    t0, t1 = ev(), ev()
    t0.record(stream)
    for _ in range(args.steps):
        last = resident_step(rec)
    t1.record(stream)
    barrier()
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    total_ms = t0.elapsed_time(t1) / args.steps
    ddim_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in rec]))
    dens_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in rec]))
    rend_ms = float(np.mean([e[2].elapsed_time(e[3]) for e in rec]))
    launches_api = (L.ssdnerf_launch_count() - launches0) / args.steps
    # kernels inside the replayed CUDA graph are launched by the driver: count the graph's kernel nodes once per replay
    graph_nodes = getattr(diffusion, '_graph_kernel_nodes', 0)
    gpu_launches = int(launches_api + graph_nodes * (DDIM_STEPS - 1))

    for _ in range(max(1, args.warmup // 2)):
        e2e_step()
    e2e_drain()
    barrier()
    s0, s1 = ev(), ev()
    s0.record(stream)
    for _ in range(args.steps):
        e2e_step()
    e2e_drain()                                        # the last gather completes inside the timed region
    s1.record(stream)
    barrier()
    e2e_ms = s0.elapsed_time(s1) / args.steps

    # ---- sample statistics of the render workload (one extra untimed launch with counts)
    code = model.code_diff_pr_inv(diffusion(model.code_diff_pr(noise), return_loss=False)).contiguous()
    _, bitfield = model.get_density(decoder, code, cfg=model.test_cfg)
    variant = decoder.fused_variant()
    cnt = R.render_fwd(variant, R.pack_planes(code, variant), (128, 128), bitfield, decoder.packed_blob(), poses=poses, intrinsics=intr,
                       img_hw=(IMG, IMG), want_blend=False)['num_samples']
    samples = int(cnt.sum().item())

    # ---- north_star's synthetic workload on EVERY rank: random-init 3x32x128x128 triplanes through the class-default decoder (variant S:
    # base 96 -> 128, colour net 144 -> 128 -> 3, xavier weights / zero bias as constructed), occupancy grid built by get_density, V views
    s_ms = s_samples = None
    if args.side_s:
        dec_s = S.build_module(dict(type='TriPlaneDecoder', max_steps=256)).to(dev).eval()
        gs = torch.Generator().manual_seed(77 + rank)
        code_s = torch.randn(B, 3, 32, 128, 128, generator=gs).clamp(-2, 2).to(dev)
        planes_s = R.pack_planes(code_s, R.DEC_S)
        _, bits_s = Dm.get_density(R.DEC_S, planes_s, (128, 128), dec_s.packed_blob(), B, density_thresh=0.1, grid_size=64, bound=1.0)

        def render_s(counts=False):
            return R.render_fwd(R.DEC_S, planes_s, (128, 128), bits_s, dec_s.packed_blob(), poses=poses, intrinsics=intr, img_hw=(IMG, IMG),
                                want_blend=True, want_counts=counts)
        s_ms = timed(render_s, args.steps, 1)
        s_samples = int(render_s(True)['num_samples'].sum().item())
        del code_s, planes_s

    # ---- strong scaling (SURVEY.md §8e secondary): ONE scene x V views, views sharded over the ranks; rank 0 owns the scene and
    # broadcasts code + bitfield (1.2 MB + 32 KB), every rank renders its contiguous view range, 8-bit images are all-gathered
    code1 = code[:1].contiguous()
    bits1 = bitfield[:1].contiguous()
    from ssdnerf_b200 import sharding as Sh
    (v_lo, v_hi), v_max = Sh.view_range(V, rank, world), Sh.max_views_per_rank(V, world)
    my_poses, my_intr = poses[:1, v_lo:v_hi].contiguous(), intr[:1, v_lo:v_hi].contiguous()
    ss_u8 = torch.zeros(v_max, IMG, IMG, 3, dtype=torch.uint8, device=dev)
    ss_all = torch.empty(world * v_max, IMG, IMG, 3, dtype=torch.uint8, device=dev)

    def strong_step():
        Sh.broadcast_scene(code1, bits1, 0)
        img, _ = model.render(decoder, code1, bits1, IMG, IMG, my_intr, my_poses, cfg=model.test_cfg)
        Sh.gather_views((img[0].clamp(0, 1) * 255.0 + 0.5).to(torch.uint8), V, out=ss_all, padded=ss_u8)
    strong_ms = timed(strong_step, args.steps, 3)

    # ---- stage-1 training step (every rank trains its own scenes; the shared decoder's gradient is all-reduced over NCCL inside the step)
    train = train2 = None
    if args.train:
        train = train_measurement(dev, timed, rank, steps=args.steps)
        train2 = train_stage2_measurement(dev, timed, rank, steps=args.steps)

    # ---- config-4 shape guided evaluations (rank 0): UNet forward + render loss forward/backward + UNet input-gradient pass
    guided = None
    if args.guided and rank == 0:
        guided = guided_measurement(dev, ev, stream, args.steps)

    # ---- reduce over ranks (max time)
    times = torch.tensor([total_ms, ddim_ms, dens_ms, rend_ms, e2e_ms, s_ms or 0.0, strong_ms, train['ms'] if train else 0.0,
                          train2['ms'] if train2 else 0.0], device=dev, dtype=torch.float64)
    sums = torch.tensor([samples, s_samples or 0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    total_ms, ddim_ms, dens_ms, rend_ms, e2e_ms, s_ms_all, strong_ms, train_ms, train2_ms = [float(x) for x in times.tolist()]
    samples_all, s_samples_all = [float(x) for x in sums.tolist()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    rays_all, trip_all = rays * world, B * world
    rays_per_s = rays_all / (rend_ms * 1e-3)
    trip_per_s = trip_all / (ddim_ms * 1e-3)
    unet_flops = UNET_FLOP_PER_SAMPLE_STEP * B * DDIM_STEPS            # per rank per step
    tf_achieved = unet_flops / (ddim_ms * 1e-3) / 1e12
    render_bytes = (samples_all / world) * RAY_GATHER_BYTES_PER_SAMPLE + rays * RAY_IO_BYTES
    kern_p = os.environ.get('SSDNERF_BENCH_KERNEL_P', 'k_render_p3')
    traffic, traffic_src = measured_traffic(kern_p, rays)
    gather_bytes = B * V * IMG * IMG * 3 * world if world > 1 else 0
    line = {
        'metric': METRIC, 'value': rays_per_s, 'unit': 'rays/s', 'triplanes_per_sec': trip_per_s,
        'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total_ms, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp16 tensor-core UNet (fp32 accumulate), fp32 renderer', 'data': 'synthetic',
        'config': {'workload': f'ssdnerf_cars_uncond (reference config, resolved): {DDIM_STEPS}-step DDIM + 8-iter density grid + {V}-view '
                               f'{IMG}x{IMG} render, batch {B}/GPU', 'global_batch': trip_all, 'rays_per_step': rays_all,
                   'samples_per_ray': samples_all / rays_all,
                   'parallelism': f'scenes x{world} (independent replicas; e2e adds the eval-side NCCL all-gather of 8-bit images)',
                   'l2_policy': 'working set per step (activations > 1 GB, 66 M rays of output) exceeds the 126 MB L2; no flush needed'},
        'stage_ms': {'ddim': ddim_ms, 'density': dens_ms, 'render': rend_ms},
        'e2e': {'value': rays_all / (e2e_ms * 1e-3), 'unit': 'rays/s', 'triplanes_per_sec': trip_all / (e2e_ms * 1e-3), 'ms_per_step': e2e_ms,
                'path': 'DiffusionNeRF.val_step: H2D (noise, poses, intrinsics) + DDIM + density + render + D2H of the images (copy stream, overlaps the next DDIM)'
                        + (' + NCCL all-gather of the 8-bit images (side stream, overlapped with the next DDIM)' if world > 1 else ''),
                'h2d_bytes_per_step': int(noise_host.numel() * 4 + poses_host.numel() * 4 + intr_host.numel() * 4),
                'd2h_bytes_per_step': int(out_host.numel() * 4), 'nccl_allgather_bytes_per_rank_per_step': int(gather_bytes)},
        'gpu_launches': gpu_launches,
        'clocks': clk,
        # dominant kernel of the step = the fused renderer (~3/4 of the step): ALGORITHMIC gather + output bytes per launch / launch
        # duration against the measured HBM copy peak (BASELINE.md 2c).  The planes (1.5 MB/scene) are L1/L2-resident, so real DRAM
        # traffic (`traffic`, from the committed ncu capture) is far below the algorithmic bytes and the binding unit is the SM.
        'roofline': {'kernel': f'{kern_p} (fused march + gather + MLP + composite), one launch per step', 'bound': 'hbm',
                     'achieved': render_bytes / (rend_ms * 1e-3) / 1e9, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                     'frac': render_bytes / (rend_ms * 1e-3) / 1e9 / pk['hbm_gbs'], 'peak_source': pk['src'] + ' (burst copy)',
                     'algorithmic_bytes_per_launch': render_bytes, 'samples_per_sec': samples_all / world / (rend_ms * 1e-3),
                     'traffic': traffic, 'traffic_source': traffic_src},
        'roofline_unet': {'kernel': 'k_gemm_tc / k_conv_row2 (tcgen05 implicit-GEMM conv / GEMM) + glue, timed as the whole DDIM stage', 'bound': 'tensor',
                          'achieved': tf_achieved, 'peak': pk['tf_sustained'], 'unit': 'TFLOP/s', 'frac': tf_achieved / pk['tf_sustained'],
                          'peak_source': f"{pk['src']} (sustained cuBLAS bf16)"},
        'strong_scaling': {'workload': f'1 scene x {V} views x {IMG}x{IMG}, views sharded over {world} rank(s); per call: broadcast code + bitfield '
                                       f'from rank 0, render, all-gather 8-bit images' if world > 1 else f'1 scene x {V} views x {IMG}x{IMG} on one GPU',
                           'ms': strong_ms, 'rays_per_sec': V * IMG * IMG / (strong_ms * 1e-3), 'scaling': 'strong'},
    }
    if s_ms is not None:
        rays_s = B * V * IMG * IMG * world
        line['render_variant_S'] = {
            'workload': f'random-init 3x32x128x128 triplanes (clamped N(0,1)), class-default TriPlaneDecoder (variant S), {B} scenes x {V} views x '
                        f'{IMG}x{IMG} per GPU, occupancy grid from get_density(thresh 0.1)', 'n_gpus': world,
            'rays_per_sec': rays_s / (s_ms_all * 1e-3), 'samples_per_sec': s_samples_all / (s_ms_all * 1e-3), 'ms': s_ms_all,
            'samples_per_ray': s_samples_all / rays_s, 'kernel': os.environ.get('SSDNERF_BENCH_KERNEL_S', 'k_render_s2'),
            'flops_per_sample': 62464, 'tflops': s_samples_all * 62464 / (s_ms_all * 1e-3) / 1e12 / world,
            'roofline': {'bound': 'hbm', 'algorithmic_bytes_per_sample': 768,
                         'achieved': (s_samples_all / world * 768 + rays * RAY_IO_BYTES) / (s_ms_all * 1e-3) / 1e9, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                         'frac': (s_samples_all / world * 768 + rays * RAY_IO_BYTES) / (s_ms_all * 1e-3) / 1e9 / pk['hbm_gbs']}}
    if guided is not None:
        line['guided'] = guided
    if train is not None:
        line['train_stage1'] = dict(train['info'], n_gpus=world, ms_per_train_step=train_ms,
                                    scenes_per_sec=train['scenes'] * world / (train_ms * 1e-3),
                                    rays_fwd_bwd_per_sec=train['rays_per_step'] * world / (train_ms * 1e-3), scaling='weak')
    if train2 is not None:
        line['train_stage2'] = dict(train2['info'], n_gpus=world, ms_per_train_step=train2_ms,
                                    triplanes_per_sec=train2['scenes'] * world / (train2_ms * 1e-3),
                                    unet_fwd_bwd_wgrad_tflops_per_gpu=3 * UNET_FLOP_PER_SAMPLE_STEP * train2['scenes'] / (train2_ms * 1e-3) / 1e12,
                                    scaling='weak')
    if args.cpu_baseline and world == 1:          # reported baseline: rank 0 at N = 1 only
        line['cpu_baseline'] = cpu_reference_sample(quick=True)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def train_measurement(dev, timed, rank, steps, views=16):
    """`stage1_cars_recons16v` (reference config, resolved) at its own sizes: samples_per_gpu scenes x 16 views 128x128 per rank,
    `extra_scene_step` code-only Adam steps + ONE joint step of latents and decoder (weight gradients from the fused backward, gradient
    all-reduce over NCCL at N > 1) per train_step, 4096 rays per scene per step, scene cache write-back included."""
    import ssdnerf_b200 as S
    cfg = reference_config('configs/paper_cfgs/stage1_cars_recons16v.py')
    train_cfg = {k: v for k, v in cfg['train_cfg'].items() if k != 'cache_load_from'}
    torch.manual_seed(0)                                   # same initial decoder on every rank (the reference broadcasts it through DDP)
    scenes = cfg['samples_per_gpu']
    model = S.build_model(dict(cfg['model'], cache_size=0), train_cfg=train_cfg, test_cfg=cfg['test_cfg']).to(dev).train()
    model.scene_cache = S.scene_cache.SceneCache(scenes, 0, 1)      # every rank caches its own `scenes` scenes
    g = torch.Generator().manual_seed(100 + rank)
    poses = orbit_poses(views)[None].repeat(scenes, 1, 1, 1).contiguous().to(dev)
    intr = torch.tensor([131.25, 131.25, 64.0, 64.0]).expand(scenes, views, 4).contiguous().to(dev)
    code = (torch.randn(scenes, 3, 6, 128, 128, generator=g) * 0.5).to(dev)
    with torch.no_grad():
        _, bits = model.get_density(model.decoder, code, cfg=dict(density_thresh=0.1))
        imgs, _ = model.render(model.decoder, code, bits, IMG, IMG, intr, poses, cfg=dict(dt_gamma_scale=0.5))
    data = dict(scene_id=list(range(scenes)), scene_name=[f'r{rank}s{i}' for i in range(scenes)], cond_imgs=imgs.clamp(0, 1), cond_poses=poses,
                cond_intrinsics=intr)
    opt = dict(decoder=torch.optim.Adam(model.decoder.parameters(), lr=1e-3))
    log = {}

    def step():
        log.update(model.train_step(data, opt)['log_vars'])
    ms = timed(step, steps, 3)
    inner = train_cfg['extra_scene_step'] + 1
    rays = scenes * (train_cfg['extra_scene_step'] * train_cfg['n_inverse_rays'] + train_cfg['n_decoder_rays'])
    if not all(v == v for v in log.values()):
        raise RuntimeError(f'stage-1 training step produced non-finite values: {log}')
    return dict(ms=ms, scenes=scenes, rays_per_step=rays,
                info={'workload': f'stage1_cars_recons16v (reference config): {scenes} scenes x {views} views {IMG}x{IMG} per GPU, {inner} optimiser '
                                  f'steps per train_step ({train_cfg["extra_scene_step"]} code-only + 1 joint with decoder-weight gradients), '
                                  f'{train_cfg["n_decoder_rays"]} rays/scene/step', 'last_log_vars': log})


def train_stage2_measurement(dev, timed, rank, steps):
    """`stage2_cars_uncond` (reference config, resolved): the denoiser (122 M parameters) trained on stored scene latents, samples_per_gpu
    scenes per rank: diffusion loss forward + UNet input / weight-gradient pass + Adam step; at N > 1 the gradient all-reduce (NCCL) is
    inside the step."""
    import ssdnerf_b200 as S
    cfg = reference_config('configs/paper_cfgs/stage2_cars_uncond.py')
    torch.manual_seed(0)
    model = S.build_model(cfg['model'], train_cfg=cfg['train_cfg'], test_cfg=cfg['test_cfg'])
    g = torch.Generator().manual_seed(0)
    for p in model.diffusion.denoising.parameters():
        if p.dim() > 1:
            p.data.copy_(torch.randn(p.shape, generator=g) * 0.02)
    model = model.to(dev).train()
    scenes = cfg['samples_per_gpu']
    g = torch.Generator().manual_seed(200 + rank)
    stored = [dict(param=dict(code=torch.tanh(torch.randn(3, 6, 128, 128, generator=g)) * 0.8, density_grid=torch.zeros(64 ** 3).half(),
                              density_bitfield=torch.zeros(64 ** 3 // 8, dtype=torch.uint8))) for _ in range(scenes)]
    data = dict(scene_id=list(range(scenes)), scene_name=[f's{i}' for i in range(scenes)], code=stored)
    opt = dict(diffusion=torch.optim.Adam(model.diffusion.parameters(), lr=1e-4))
    log = {}

    def step():
        log.update(model.train_step(data, opt)['log_vars'])
    ms = timed(step, steps, 3)
    if not all(v == v for v in log.values()):
        raise RuntimeError(f'stage-2 training step produced non-finite values: {log}')
    return dict(ms=ms, scenes=scenes,
                info={'workload': f'stage2_cars_uncond (reference config): {scenes} stored scenes per GPU, diffusion loss + UNet forward / input-gradient / '
                                  f'weight-gradient pass + Adam on 122 M parameters', 'last_log_vars': {k: v for k, v in log.items() if 'quartile' not in k}})


def guided_measurement(dev, ev, stream, steps, scenes=8, evals=6):
    """BASELINE config 4 (`ssdnerf_chairs_recons1v`, reference config resolved): `steps` val_guide calls of `evals` guided x_0 predictions
    each at 8 scenes x one 128x128 conditioning view = what every DDIM / langevin step of val_guide costs (445 of them per batch in the
    shipped config)."""
    model, _ = build_model(dev, seed=1, rel='configs/paper_cfgs/ssdnerf_chairs_recons1v.py')
    diffusion, decoder = model.diffusion_ema, model.decoder_ema
    g = torch.Generator().manual_seed(5)
    code0 = (torch.randn(scenes, 3, 6, 128, 128, generator=g) * 0.5).to(dev)
    poses = orbit_poses(4)[None].repeat(scenes, 1, 1, 1)[:, :1].contiguous().to(dev)
    intr = torch.tensor([131.25, 131.25, 64.0, 64.0]).expand(scenes, 1, 4).contiguous().to(dev)
    with torch.no_grad():
        _, bits0 = model.get_density(decoder, code0, cfg=dict(density_thresh=0.1))
        img0, _ = model.render(decoder, code0, bits0, IMG, IMG, intr, poses, cfg=model.test_cfg)
    data = dict(cond_imgs=img0, cond_intrinsics=intr, cond_poses=poses, noise=torch.randn(scenes, 3, 6, 128, 128, generator=g).to(dev))
    # time `evals` guided evaluations through the public sampler: num_timesteps = evals, no langevin
    model.test_cfg.update(num_timesteps=evals, langevin_steps=0)
    diffusion.test_cfg.update(num_timesteps=evals, langevin_steps=0)
    model.val_guide(data)                                  # warm-up (packs the transposed weights, sizes the scratch)
    torch.cuda.synchronize(dev)
    a, b = ev(), ev()
    a.record(stream)
    for _ in range(steps):
        model.val_guide(data)
    b.record(stream)
    torch.cuda.synchronize(dev)
    ms = a.elapsed_time(b) / (evals * steps)
    return {'workload': f'ssdnerf_chairs_recons1v (reference config): {scenes} scenes, 1 cond view {IMG}x{IMG}, grad_through_unet (default), '
                        f'{steps} val_guide calls of {evals} guided evaluations', 'ms_per_guided_eval': ms, 'guided_evals_per_sec': 1e3 / ms,
            'rays_fwd_bwd_per_sec': scenes * IMG * IMG / (ms * 1e-3),
            'unet_fwd_bwd_tflops': 3 * UNET_FLOP_PER_SAMPLE_STEP * scenes / (ms * 1e-3) / 1e12,
            'note': 'flops = forward + data-gradient pass (2x forward) of the UNet only; includes the occupancy update and the fused render loss'}


# ----------------------------------------------------------------------------------------------------------- reference arm
def usable_cores():
    """host cores this process may really use: affinity mask capped by the cgroup CPU quota (a 128-thread pool on an
    8-core quota is ~100x slower than 8 threads)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, min(n, 64))


def cpu_reference_sample(quick=False, unet_evals=4, views=4):
    """Reference arithmetic on the host cores = the oracle port (PyTorch-CPU UNet + C marcher/compositor + PyTorch-CPU decode);
    the reference itself has no CPU path for the renderer (SURVEY.md F3). Bounded sample of the bench workload:
    B=1 scene, `unet_evals` UNet evaluations (extrapolated x50/`unet_evals`), `views` 128x128 views."""
    from oracle import render_port as rp
    from oracle import unet_port as up
    cores = usable_cores()
    torch.set_num_threads(cores)
    if quick:
        unet_evals, views = 2, 1
    spec = up.unet_spec()
    sd = up.random_state_dict(spec, seed=0)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 18, 128, 128, generator=g)
    t = torch.tensor([999])
    with torch.no_grad():
        up.unet_forward(sd, spec, x, t)                 # warm-up
        t0 = time.perf_counter()
        for _ in range(unet_evals):
            v = up.unet_forward(sd, spec, x, t)
        t_unet = (time.perf_counter() - t0) / unet_evals
    params = rp.make_decoder_params('P', 0, nonzero_dir=False)
    code = torch.randn(1, 3, 6, 128, 128, generator=g).clamp(-2, 2)
    rands = [torch.rand(64 ** 3, 3, generator=g)]
    _, bf = rp.get_density(params, code, rands, density_thresh=0.1)
    poses = orbit_poses(NUM_VIEWS)[:views]
    intr = torch.tensor([131.25, 131.25, 64.0, 64.0]).expand(views, 4).contiguous()
    t0 = time.perf_counter()
    rp.render_image(params, code[0], bf[0], poses, intr, IMG, IMG, max_steps=256)
    t_render = time.perf_counter() - t0
    rays = views * IMG * IMG
    return {'value': rays / t_render, 'unit': 'rays/s', 'triplanes_per_sec': 1.0 / (t_unet * DDIM_STEPS), 'cores': cores, 'kind': 'port',
            'sample': f'B=1: {unet_evals} UNet evaluations (fp32, {t_unet:.3f} s each, x{DDIM_STEPS} extrapolated) + {views} view(s) '
                      f'{IMG}x{IMG} through the oracle host loop ({t_render:.2f} s)',
            'unet_s_per_eval': t_unet, 'render_s': t_render}


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    vals, trips, t_all = [], [], []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = cpu_reference_sample(unet_evals=8, views=8)
        if i >= args.warmup:
            vals.append(r['value']); trips.append(r['triplanes_per_sec']); t_all.append(time.perf_counter() - t0)
    v, tr = float(np.mean(vals)), float(np.mean(trips))
    r['value'] = v
    r['triplanes_per_sec'] = tr
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'rays/s', 'triplanes_per_sec': tr, 'n_gpus': int(os.environ.get('WORLD_SIZE', 1)),
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': float(np.mean(t_all)) * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
            'config': {'workload': f'ssdnerf_cars_uncond: {DDIM_STEPS}-step DDIM + {IMG}x{IMG} render, bounded CPU sample of the same workload (see cpu_baseline.sample)'},
            'cpu_baseline': r, 'e2e': {'value': v, 'unit': 'rays/s', 'triplanes_per_sec': tr, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=B_PER_GPU)
    ap.add_argument('--views', type=int, default=NUM_VIEWS)
    ap.add_argument('--no-cpu-baseline', dest='cpu_baseline', action='store_false')
    ap.add_argument('--no-side-s', dest='side_s', action='store_false', help='skip the variant-S renderer workload')
    ap.add_argument('--no-guided', dest='guided', action='store_false', help='skip the config-4 guided-evaluation measurement')
    ap.add_argument('--no-train', dest='train', action='store_false', help='skip the stage-1 training-step measurement')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the last timed step\'s triplanes, density grid / bitfield, images and '
                    'depths as DIR/<name>.npy (float32; arrays beyond a 64 MB total are written as a seeded sample)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of --impl b200')
    if args.warmup < 3 and args.impl == 'b200':
        args.warmup = 3      # timing rule: at least 3 warm-up steps
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
