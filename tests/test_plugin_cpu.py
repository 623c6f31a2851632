"""Plugin surface on CPU: registry names, config loading, state-dict keys, host-side DDIM tables (no GPU compute)."""
import os

import numpy as np
import pytest
import torch

import ssdnerf_b200 as S
from oracle import unet_port as up

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE_CONFIGS = os.path.join(ROOT, 'tests', 'golden', 'reference_configs.json')


def test_registry_names():
    for n in ('TriPlaneDecoder', 'GaussianDiffusion', 'DenoisingUnetMod', 'TanhCode', 'IdentityCode', 'NormalizedTanhCode', 'MSELoss', 'RegLoss', 'TVLoss',
              'DDPMMSELossMod', 'SNRWeightedTimeStepSampler', 'UniformTimeStepSamplerMod'):
        assert n in S.MODULES
    assert 'DiffusionNeRF' in S.MODELS and 'MultiSceneNeRF' in S.MODELS


def test_build_from_repo_config_and_state_dict_keys():
    cfg = S.Config.fromfile(os.path.join(ROOT, 'configs', 'cars_uncond_b200.py'))
    m = S.build_model(cfg.model, test_cfg=cfg.test_cfg)
    sd = m.diffusion.denoising.state_dict()
    ref = up.random_state_dict(up.unet_spec())
    assert set(sd) == set(ref) and all(sd[k].shape == ref[k].shape for k in ref)
    assert sum(v.numel() for v in sd.values()) == 122434194
    dec = m.decoder.state_dict()
    assert tuple(dec['base_net.0.weight'].shape) == (64, 18) and tuple(dec['dir_net.0.weight'].shape) == (64, 16)
    assert tuple(dec['color_net.0.weight'].shape) == (3, 64) and tuple(dec['aabb'].shape) == (6,)
    # EMA twins selected at inference exist (diffusion_nerf.py:192-193)
    assert hasattr(m, 'decoder_ema') and hasattr(m, 'diffusion_ema')
    assert m.code_diff_pr(torch.zeros(2, 3, 6, 128, 128)).shape == (2, 18, 128, 128)
    assert m.code_diff_pr_inv(torch.zeros(2, 18, 128, 128)).shape == (2, 3, 6, 128, 128)


@pytest.mark.parametrize('cfg_rel', ['configs/paper_cfgs/ssdnerf_cars_uncond.py', 'configs/paper_cfgs/ssdnerf_chairs_recons1v.py',
                                     'configs/paper_cfgs/ssdnerf_abotables_uncond.py'])
def test_reference_configs_build_unchanged(cfg_rel, tmp_path):
    """the reference's config as resolved into tests/golden/reference_configs.json (tests/golden/make_config_fixtures.py), loaded back
    through Config.fromfile from a `_base_` file and a file overriding its test_cfg, as the reference composes its configs"""
    import json
    ref = json.load(open(REFERENCE_CONFIGS))[cfg_rel]
    (tmp_path / 'base.py').write_text(f"model = {ref['model']!r}\ntrain_cfg = {ref['train_cfg']!r}\ntest_cfg = dict(num_timesteps=-1)\n")
    (tmp_path / 'cfg.py').write_text(f"_base_ = 'base.py'\ntest_cfg = {ref['test_cfg']!r}\n")
    cfg = S.Config.fromfile(str(tmp_path / 'cfg.py'))
    assert json.loads(json.dumps(cfg)) == {k: ref[k] for k in ('model', 'train_cfg', 'test_cfg')}
    m = S.build_model(cfg.model, train_cfg=cfg.get('train_cfg'), test_cfg=cfg.get('test_cfg'))
    assert type(m).__name__ == 'DiffusionNeRF'
    assert m.diffusion.test_cfg['num_timesteps'] == cfg.test_cfg['num_timesteps']


def test_every_reference_config_builds_from_the_fixture():
    """tests/golden/reference_configs.json = every config the reference ships, resolved (tests/golden/make_config_fixtures.py); each one
    builds through the registry unchanged"""
    import json
    cfgs = json.load(open(REFERENCE_CONFIGS))
    assert len(cfgs) == 24
    for name, c in cfgs.items():
        m = S.build_model(c['model'], train_cfg=c['train_cfg'], test_cfg=c['test_cfg'])
        assert type(m).__name__ in ('DiffusionNeRF', 'MultiSceneNeRF'), name
    # the bench / GPU-test config is the fixture entry, and the repo's restated config file agrees with it
    own = S.Config.fromfile(os.path.join(ROOT, 'configs', 'cars_uncond_b200.py'))
    refc = cfgs['configs/paper_cfgs/ssdnerf_cars_uncond.py']
    for k in ('code_size', 'code_reshape', 'grid_size', 'decoder_use_ema', 'bg_color'):
        assert json.loads(json.dumps(own.model[k])) == refc['model'][k], k
    assert json.loads(json.dumps(own.model['decoder'])) == refc['model']['decoder']
    assert json.loads(json.dumps(own.model['diffusion']['denoising'])) == refc['model']['diffusion']['denoising']
    assert json.loads(json.dumps(dict(own.test_cfg))) == refc['test_cfg']


def test_code_activations_scene_io_and_losses(tmp_path):
    from ssdnerf_b200.nerf import BaseNeRF, NormalizedTanhCode, TanhCode, TVLoss
    act = NormalizedTanhCode(mean=0.0, std=0.5, clip_range=2)
    act.running_mean.fill_(0.1); act.running_var.fill_(0.3)
    x = torch.linspace(-1.5, 1.5, 31)
    torch.testing.assert_close(act.inverse(act(x)), x, rtol=1e-4, atol=1e-4)
    # formula of base_nerf.py:65-76
    scale = 0.5 / (0.3 ** 0.5 + 1e-5)
    torch.testing.assert_close(act(x), torch.tanh((x * scale + (0.0 - 0.1 * scale)) / 2) * 2)
    assert set(act.state_dict()) == {'running_mean', 'running_var'}
    act.train()
    before = act.running_mean.clone()
    act(x, update_stats=True)
    assert not torch.equal(before, act.running_mean)
    # save_scene / load_scene round trip in the reference's file format (base_nerf.py:141-170)
    code = torch.randn(2, 3, 6, 8, 8)
    grid = torch.rand(2, 64).half()
    bits = torch.randint(0, 255, (2, 8), dtype=torch.uint8)
    BaseNeRF.save_scene(str(tmp_path), code, grid, bits, ['a', 'b'])
    states = [torch.load(os.path.join(tmp_path, n + '.pth')) for n in ('a', 'b')]
    assert set(states[0]) == {'scene_name', 'param'} and set(states[0]['param']) == {'code', 'density_grid', 'density_bitfield'}
    holder = torch.nn.Module.__new__(BaseNeRF); torch.nn.Module.__init__(holder)
    holder.code_activation = TanhCode(scale=2); holder.register_buffer('_p', torch.zeros(1)); holder.register_parameter('w', torch.nn.Parameter(torch.zeros(1)))
    c2, g2, b2 = BaseNeRF.load_scene(holder, dict(code=states), load_density=True)
    assert torch.equal(c2, code) and torch.equal(g2, grid) and torch.equal(b2, bits)
    pre = dict(param=dict(code_=torch.randn(3, 6, 8, 8)))             # training-cache states hold the pre-activation latent
    c3, _, _ = BaseNeRF.load_scene(holder, dict(code=[pre]))
    torch.testing.assert_close(c3[0], pre['param']['code_'].tanh() * 2)
    assert float(TVLoss(power=1.5)(torch.ones(1, 3, 6, 8, 8))) == 0.0


def test_ddim_tables_match_oracle():
    from ssdnerf_b200.diffusion import GaussianDiffusion
    from ssdnerf_b200.unet import DenoisingUnetMod
    unet = DenoisingUnetMod(image_size=32, in_channels=18, base_channels=64, channels_cfg=[1, 2], resblocks_per_downsample=1,
                            num_heads=2, attention_res=[16], use_scale_shift_norm=True)
    d = GaussianDiffusion(unet, betas_cfg=dict(type='linear'), test_cfg=dict(num_timesteps=50))
    dv = up.diffusion_vars(up.linear_betas())
    np.testing.assert_array_equal(d.alphas_bar, dv['alphas_bar'])
    np.testing.assert_array_equal(d.tilde_betas_t, dv['tilde_betas_t'])
    ts = d.ddim_timesteps(50)
    assert ts[0] == 999 and ts[-1] == 19 and len(ts) == 50
    coef = d.ddim_coefficients(ts)
    assert coef.shape == (50, 4) and coef[-1, 2] == 1.0          # alpha_bar_prev = 1 at the last step (t_prev = -1)
    # time embedding of the module equals the oracle restatement
    sd = {k: v.clone() for k, v in unet.state_dict().items()}
    e1 = unet.embedding(ts)
    e2 = up.time_embedding(sd, ts.float(), 64)
    torch.testing.assert_close(e1, e2)


def test_unsupported_paths_fail_loudly():
    cfg = S.Config.fromfile(os.path.join(ROOT, 'configs', 'cars_uncond_b200.py'))
    m = S.build_model(cfg.model, test_cfg=cfg.test_cfg)
    # training runs on the native kernels only: CPU tensors are refused, never routed to a PyTorch fallback
    stored = [dict(param=dict(code=torch.zeros(3, 6, 128, 128), density_grid=torch.zeros(64 ** 3).half(),
                              density_bitfield=torch.zeros(64 ** 3 // 8, dtype=torch.uint8)))]
    m.train_cfg = dict()
    with pytest.raises(S._lib.SSDNeRFNativeError):
        m.train().train_step(dict(scene_id=[0], scene_name=['a'], code=stored), dict(diffusion=torch.optim.SGD(m.diffusion.parameters(), lr=0.1)))
    m.eval()
    with pytest.raises(S._lib.SSDNeRFNativeError):
        m.render(m.decoder, torch.zeros(1, 3, 6, 128, 128), torch.zeros(1, 32768, dtype=torch.uint8), 8, 8,
                 torch.zeros(1, 1, 4), torch.zeros(1, 1, 4, 4))


def test_guidance_host_logic():
    """ray batches, loss modules, activations: the host-side pieces of the guided path (base_nerf.py:231-296) on CPU tensors"""
    from ssdnerf_b200.nerf import DiffusionNeRF, MSELoss, RegLoss, TanhCode
    from ssdnerf_b200.activation import trunc_exp
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(2, 3, 8, 8, 3, generator=g)                    # 2 scenes x 3 views x 8x8
    ro, rd = torch.rand(2, 3, 8, 8, 3, generator=g), torch.rand(2, 3, 8, 8, 3, generator=g)
    inds, nb = DiffusionNeRF.get_raybatch_inds(imgs, 50)
    assert nb == 4 and [i.shape for i in inds] == [(2, 50), (2, 50), (2, 50), (2, 42)]
    allidx = torch.cat(list(inds), dim=1)
    assert all(torch.equal(torch.sort(allidx[s]).values, torch.arange(192)) for s in range(2))      # a permutation per scene
    o, d, t = DiffusionNeRF.ray_sample(ro, rd, imgs, 50, sample_inds=inds[1])
    assert o.shape == (2, 50, 3) and torch.equal(t[1], imgs.reshape(2, -1, 3)[1][inds[1][1]]) and torch.equal(d[0], rd.reshape(2, -1, 3)[0][inds[1][0]])
    assert DiffusionNeRF.get_raybatch_inds(imgs, 192) == (None, None)                                # whole image fits: no sampling
    o2, _, t2 = DiffusionNeRF.ray_sample(ro, rd, imgs, 4096)
    assert o2.shape == (2, 192, 3) and torch.equal(t2, imgs.reshape(2, -1, 3))
    a, b = torch.rand(5, 3, generator=g), torch.rand(5, 3, generator=g)
    torch.testing.assert_close(MSELoss(loss_weight=20.0)(a, b), ((a - b) ** 2).mean() * 20.0)
    torch.testing.assert_close(RegLoss(power=2, loss_weight=3e-3)(a), (a ** 2).mean() * 3e-3)
    torch.testing.assert_close(RegLoss(power=1)(a - 0.5), (a - 0.5).abs().mean())
    tc = TanhCode(scale=2)
    x = torch.linspace(-3, 3, 13)
    torch.testing.assert_close(tc.inverse(tc(x)), x, rtol=1e-4, atol=1e-4)
    z = torch.tensor([-30.0, 0.5, 30.0], requires_grad=True)
    trunc_exp(z).sum().backward()
    torch.testing.assert_close(z.grad, torch.tensor([1e-6, float(np.exp(0.5)), 1e6]))


def test_guided_sampling_contract():
    """guidance through the denoiser runs on the native UNet (forward + input-gradient pass): CPU tensors never reach a fallback"""
    cfg = S.Config.fromfile(os.path.join(ROOT, 'configs', 'cars_uncond_b200.py'))
    m = S.build_model(cfg.model, test_cfg=dict(cfg.test_cfg))
    d = m.diffusion
    with pytest.raises(S._lib.SSDNeRFNativeError):
        d.pred_x_0(torch.zeros(1, 18, 128, 128), torch.tensor([10]), grad_guide_fn=lambda x: x.sum(), cfg=dict(clip_range=[-2, 2]))
    with pytest.raises(S._lib.SSDNeRFNativeError):
        m.val_guide(dict(cond_imgs=torch.zeros(1, 1, 8, 8, 3), cond_intrinsics=torch.ones(1, 1, 4), cond_poses=torch.eye(4).expand(1, 1, 4, 4)))
    with pytest.raises(S._lib.SSDNeRFNativeError):
        m.val_optim(dict(cond_imgs=torch.zeros(1, 1, 8, 8, 3), cond_intrinsics=torch.ones(1, 1, 4), cond_poses=torch.eye(4).expand(1, 1, 4, 4)))
    # the step-wise sampler is selected for guidance / langevin / eta > 0 and refuses image-conditioned denoisers
    with pytest.raises(NotImplementedError, match='concat_cond'):
        d._ddim_sample_stepwise(torch.zeros(1, 18, 128, 128), concat_cond=torch.zeros(1, 1, 3, 128, 128))
