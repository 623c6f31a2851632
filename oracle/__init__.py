"""CPU oracle for the SSDNeRF hot paths -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package; ``ssdnerf_b200`` never does.

PARITY UNPINNED BY REFERENCE TESTS: Lakonik/SSDNeRF ships no test-suite, golden
vectors or CPU path for these kernels (SURVEY.md F2/F3).  The GPU kernels the
tests hold to this restatement are in turn compared with the outputs of the
reference's own CUDA kernels (built into ``oracle/_ref`` by ``oracle/build_ref.sh``),
stored in ``tests/golden/reference_kernels_v1.npz`` (``tests/test_ref_gpu.py``).

``lib()`` returns the ctypes handle of ``oracle/_build/liboracle.so`` (compiled
from ``ssdnerf_oracle.c`` with gcc on first use).
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, 'ssdnerf_oracle.c')
_OUT = os.path.join(_HERE, '_build', 'liboracle.so')
_LIB = None


def build(force=False):
    """gcc -O2 -ffp-contract=off: every FMA in the oracle is an explicit fmaf()."""
    if not force and os.path.exists(_OUT) and os.path.getmtime(_OUT) >= os.path.getmtime(_SRC):
        return _OUT
    os.makedirs(os.path.dirname(_OUT), exist_ok=True)
    cmd = ['gcc', '-O2', '-std=c11', '-fPIC', '-shared', '-ffp-contract=off', '-fno-fast-math',
           '-fvisibility=hidden', '-o', _OUT, _SRC, '-lm']
    subprocess.check_call(cmd)
    return _OUT


def lib():
    global _LIB
    if _LIB is None:
        _LIB = ctypes.CDLL(build())
    return _LIB


def _p(a, ct=None):
    if a is None:
        return None
    assert a.flags['C_CONTIGUOUS']
    return a.ctypes.data_as(ctypes.c_void_p)


F32 = np.float32
I32 = np.int32
U8 = np.uint8
c_u32 = ctypes.c_uint32
c_f32 = ctypes.c_float


def near_far_from_aabb(rays_o, rays_d, aabb, min_near=0.2):
    rays_o = np.ascontiguousarray(rays_o, F32).reshape(-1, 3)
    rays_d = np.ascontiguousarray(rays_d, F32).reshape(-1, 3)
    aabb = np.ascontiguousarray(aabb, F32)
    N = rays_o.shape[0]
    nears = np.empty(N, F32)
    fars = np.empty(N, F32)
    lib().orc_near_far_from_aabb(_p(rays_o), _p(rays_d), _p(aabb), c_u32(N), c_f32(min_near), _p(nears), _p(fars))
    return nears, fars


def morton3D(coords):
    coords = np.ascontiguousarray(coords, I32).reshape(-1, 3)
    out = np.empty(coords.shape[0], I32)
    lib().orc_morton3D(_p(coords), c_u32(coords.shape[0]), _p(out))
    return out


def morton3D_invert(indices):
    indices = np.ascontiguousarray(indices, I32).reshape(-1)
    out = np.empty((indices.shape[0], 3), I32)
    lib().orc_morton3D_invert(_p(indices), c_u32(indices.shape[0]), _p(out))
    return out


def packbits(grid, thresh):
    grid = np.ascontiguousarray(grid, F32)
    N = grid.size // 8
    out = np.empty(N, U8)
    lib().orc_packbits(_p(grid), c_u32(N), c_f32(float(thresh)), _p(out))
    return out


def march_rays(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, bound, bitfield, C, H, nears, fars,
               align=-1, dt_gamma=0.0, max_steps=1024, noises=None, return_voxels=False):
    """Mirror of lib/ops/raymarching/raymarching.py:402-460 (`_march_rays.forward`)."""
    M = n_alive * n_step
    if align > 0:
        M += align - (M % align)
    xyzs = np.zeros((M, 3), F32)
    dirs = np.zeros((M, 3), F32)
    deltas = np.zeros((M, 2), F32)
    vox = np.full(M, -1, I32) if return_voxels else None
    noises = np.zeros(n_alive, F32) if noises is None else np.ascontiguousarray(noises, F32)
    lib().orc_march_rays(c_u32(n_alive), c_u32(n_step), _p(rays_alive), _p(rays_t), _p(rays_o), _p(rays_d),
                         c_f32(bound), c_f32(dt_gamma), c_u32(max_steps), c_u32(C), c_u32(H), _p(bitfield),
                         _p(nears), _p(fars), _p(xyzs), _p(dirs), _p(deltas), _p(noises), _p(vox))
    if return_voxels:
        return xyzs, dirs, deltas, vox
    return xyzs, dirs, deltas


def composite_rays(n_alive, n_step, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image, T_thresh=1e-2):
    sigmas = np.ascontiguousarray(sigmas, F32)
    rgbs = np.ascontiguousarray(rgbs, F32)
    lib().orc_composite_rays(c_u32(n_alive), c_u32(n_step), c_f32(T_thresh), _p(rays_alive), _p(rays_t),
                             _p(sigmas), _p(rgbs), _p(deltas), _p(weights_sum), _p(depth), _p(image))


def march_rays_train(rays_o, rays_d, bound, bitfield, C, H, nears, fars, dt_gamma=0.0, max_steps=1024,
                     noises=None, align=-1, return_voxels=False):
    """Mirror of `_march_rays_train.forward` (raymarching.py:200-285) with force_all_rays=True;
    point offsets are the deterministic prefix sum (reference order is atomicAdd arrival)."""
    rays_o = np.ascontiguousarray(rays_o, F32).reshape(-1, 3)
    rays_d = np.ascontiguousarray(rays_d, F32).reshape(-1, 3)
    N = rays_o.shape[0]
    rays = np.empty((N, 3), I32)
    counter = np.zeros(2, I32)
    noises = np.zeros(N, F32) if noises is None else np.ascontiguousarray(noises, F32)
    args = lambda xyzs, dirs, deltas, M, vox: (
        _p(rays_o), _p(rays_d), _p(bitfield), c_f32(bound), c_f32(dt_gamma), c_u32(max_steps), c_u32(N), c_u32(C),
        c_u32(H), c_u32(M), _p(nears), _p(fars), _p(xyzs), _p(dirs), _p(deltas), _p(rays), _p(counter), _p(noises), _p(vox))
    lib().orc_march_rays_train(*args(None, None, None, 0, None))
    m = int(counter[0])
    M = m
    if align > 0:
        M += align - M % align
    xyzs = np.zeros((M, 3), F32)
    dirs = np.zeros((M, 3), F32)
    deltas = np.zeros((M, 2), F32)
    vox = np.full(M, -1, I32) if return_voxels else None
    counter[:] = 0
    lib().orc_march_rays_train(*args(xyzs, dirs, deltas, M, vox))
    if return_voxels:
        return xyzs, dirs, deltas, rays, vox
    return xyzs, dirs, deltas, rays


def composite_rays_train_forward(sigmas, rgbs, deltas, rays, T_thresh=1e-4):
    sigmas = np.ascontiguousarray(sigmas, F32)
    rgbs = np.ascontiguousarray(rgbs, F32)
    M, N = sigmas.shape[0], rays.shape[0]
    ws = np.empty(N, F32)
    depth = np.empty(N, F32)
    image = np.empty((N, 3), F32)
    lib().orc_composite_rays_train_forward(_p(sigmas), _p(rgbs), _p(deltas), _p(rays), c_u32(M), c_u32(N),
                                           c_f32(T_thresh), _p(ws), _p(depth), _p(image))
    return ws, depth, image


def composite_rays_train_backward(grad_ws, grad_image, sigmas, rgbs, deltas, rays, ws, image, T_thresh=1e-4):
    sigmas = np.ascontiguousarray(sigmas, F32)
    rgbs = np.ascontiguousarray(rgbs, F32)
    grad_ws = np.ascontiguousarray(grad_ws, F32)
    grad_image = np.ascontiguousarray(grad_image, F32)
    M, N = sigmas.shape[0], rays.shape[0]
    gs = np.zeros(M, F32)
    gc = np.zeros((M, 3), F32)
    lib().orc_composite_rays_train_backward(_p(grad_ws), _p(grad_image), _p(sigmas), _p(rgbs), _p(deltas), _p(rays),
                                            _p(ws), _p(image), c_u32(M), c_u32(N), c_f32(T_thresh), _p(gs), _p(gc))
    return gs, gc


def sh_encode(dirs, degree=4):
    dirs = np.ascontiguousarray(dirs, F32).reshape(-1, 3)
    out = np.empty((dirs.shape[0], degree * degree), F32)
    lib().orc_sh_encode(_p(dirs), c_u32(dirs.shape[0]), c_u32(degree), _p(out))
    return out


def trace_rays(rays_o, rays_d, nears, fars, bound, bitfield, C, H, dt_gamma=0.0, max_steps=256, cap=None):
    """Integer trace: per ray the occupancy-bit index of each sample it would take (no T early-exit)."""
    rays_o = np.ascontiguousarray(rays_o, F32).reshape(-1, 3)
    rays_d = np.ascontiguousarray(rays_d, F32).reshape(-1, 3)
    N = rays_o.shape[0]
    cap = cap or (max_steps + 7)
    trace = np.empty((N, cap), I32)
    ts = np.empty((N, cap), F32)
    counts = np.empty(N, I32)
    lib().orc_trace_rays(_p(rays_o), _p(rays_d), _p(nears), _p(fars), c_u32(N), c_f32(bound), c_f32(dt_gamma),
                         c_u32(max_steps), c_u32(C), c_u32(H), _p(bitfield), c_u32(cap), _p(trace), _p(ts), _p(counts))
    return trace, ts, counts
