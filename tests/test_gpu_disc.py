"""GPU parity of the discriminator realism term (reference calc_loss_disc, util_latent_aug.py:363-371)
against the CPU oracle (oracle/sg2_disc.py + autograd): logits, loss, the gradient back to the image, and the
full loop with w_disc > 0.  The discriminator runs in the engine's precision:
  * fp32_parity (split-bf16 operands): logits / loss 1e-4, input gradient rel-L2 5e-3 (measured 1e-5 .. 1.6e-3: a single
    sign flip of a near-zero pre-activation is visible at the 1e-3 level), loop with the
    term 1e-3 on final w and image (measured ~1e-5) -- the north_star tolerance
  * bf16: logits 2e-2 (max error / max |logit|), loss 1e-2; bf16 rounding alone moves the input gradient of a
    random-init D by ~5 % (sign flips of near-zero pre-activations, each changing that unit's gradient factor from 1
    to 0.2; measured on the oracle with ``emulate_bf16``), so the bf16 gradient is checked in direction and size only
    (cosine > 0.99, rel-L2 < 0.15 against both the fp32 and the bf16-emulating oracle; 0.2 with the clamp engaged, whose
    hi-plane window adds up to 6e-2, tests/test_gpu_act_clamp.py); loop with the term 1e-2.
"""
import random

import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu

TOL = {'fp32_parity': 1e-3, 'bf16': 1e-2}


def _setup(cfg, precision, noise_strength=0.1, conv_clamp=256.0, mbstd_group_size=4):
    """G and D with the same conv_clamp (the clamp engages at 1.0 / 0.7, tests/test_gpu_act_clamp.py)."""
    from latentaugment_b200.engine import SynthesisEngine
    from oracle import sg2_disc, synthetic
    wl = synthetic.make_workload(cfg, noise_strength=noise_strength, conv_clamp=conv_clamp)
    G, c = wl['G'], wl['cfg']
    D = sg2_disc.make_discriminator(img_resolution=c['img_resolution'], img_channels=c['img_channels'], channel_base=c['channel_base'],
                                    channel_max=c['channel_max'], conv_clamp=conv_clamp, mbstd_group_size=mbstd_group_size)
    eng = SynthesisEngine(dict(G.state_dict()), img_resolution=G.img_resolution, img_channels=G.img_channels,
                          w_dim=G.w_dim, z_dim=G.z_dim, conv_clamp=conv_clamp, batch=wl['w0'].shape[0], precision=precision)
    eng.set_discriminator(dict(D.state_dict()), conv_clamp=conv_clamp, mbstd_group_size=mbstd_group_size)
    return wl, D, eng


# (cfg, conv_clamp, mbstd_group_size): the default networks under their plain ids, the clamp off / engaged
# (tests/test_gpu_act_clamp.py) and the paper256 / paper512 minibatch-stddev group of 8 (batch 8: tiny128)
DISC_CASES = ([pytest.param(c, 256.0, 4, id=c) for c in ('tiny', 'tiny128', 'small')]
              + [pytest.param(c, v, 4, id=f'{c}-clamp{v}') for c in ('tiny', 'small') for v in (None, 1.0, 0.7)]
              + [pytest.param('tiny128', v, 8, id=f'tiny128-clamp{v}-mbstd8') for v in (256.0, 0.7)])


@pytest.mark.parametrize('cfg,conv_clamp,mbstd', DISC_CASES)
def test_disc_fp32_parity_logits_loss_and_gradient(cfg, conv_clamp, mbstd):
    wl, D, eng = _setup(cfg, 'fp32_parity', conv_clamp=conv_clamp, mbstd_group_size=mbstd)
    c = wl['cfg']
    B = wl['w0'].shape[0]
    x = (torch.rand([B, c['img_channels'], c['img_resolution'], c['img_resolution']], generator=torch.Generator().manual_seed(11)) * 2 - 1)
    x = x.requires_grad_(True)
    logits_ref = D(x, c=None)
    loss_ref = torch.nn.functional.softplus(-logits_ref).mean() * 0.7
    loss_ref.backward()
    logits = eng.disc_logits(x).cpu()
    loss, grad = eng.disc_loss_grad(x, w_disc=0.7)
    eng.debug_check()
    el = float((logits - logits_ref.detach()).abs().max() / logits_ref.detach().abs().max())
    eg = rel_l2(grad.cpu(), x.grad)
    print(f'\n[disc fp32_parity {cfg} conv_clamp={conv_clamp} mbstd={mbstd}] logits max-rel={el:.3e} loss ours={float(loss):.7f} oracle={float(loss_ref.detach()):.7f} grad rel_l2={eg:.3e}')
    assert el < 1e-4
    assert abs(float(loss) - float(loss_ref.detach())) < 1e-4 * abs(float(loss_ref.detach()))
    assert eg < 5e-3          # one flipped near-zero pre-activation among ~3e5 units is already ~1.5e-3


@pytest.mark.parametrize('cfg,conv_clamp,mbstd', DISC_CASES)
def test_disc_logits_loss_and_gradient(cfg, conv_clamp, mbstd):
    wl, D, eng = _setup(cfg, 'bf16', conv_clamp=conv_clamp, mbstd_group_size=mbstd)
    c = wl['cfg']
    B = wl['w0'].shape[0]
    x = (torch.rand([B, c['img_channels'], c['img_resolution'], c['img_resolution']], generator=torch.Generator().manual_seed(11)) * 2 - 1)
    x = x.requires_grad_(True)
    logits_ref = D(x, c=None)
    loss_ref = torch.nn.functional.softplus(-logits_ref).mean() * 0.7
    loss_ref.backward()
    g_ref = x.grad.clone()
    from oracle import sg2_disc
    sg2_disc.Conv2dLayer.emulate_bf16 = True
    try:
        x.grad = None
        (torch.nn.functional.softplus(-D(x, c=None)).mean() * 0.7).backward()
        g_emul = x.grad.clone()
    finally:
        sg2_disc.Conv2dLayer.emulate_bf16 = False
    logits = eng.disc_logits(x).cpu()
    loss, grad = eng.disc_loss_grad(x, w_disc=0.7)
    eng.debug_check()
    grad = grad.cpu()
    el = float((logits - logits_ref.detach()).abs().max() / logits_ref.detach().abs().max())
    eg, ee = rel_l2(grad, g_ref), rel_l2(grad, g_emul)
    cos = float((grad.double() * g_ref.double()).sum() / grad.double().norm() / g_ref.double().norm())
    print(f'\n[disc {cfg} conv_clamp={conv_clamp} mbstd={mbstd}] logits max-rel={el:.3e} loss ours={float(loss):.6f} oracle={float(loss_ref.detach()):.6f} '
          f'grad rel_l2 vs fp32 oracle={eg:.3e} (cos {cos:.5f}), vs bf16-emulating oracle={ee:.3e}')
    assert el < 2e-2
    assert abs(float(loss) - float(loss_ref.detach())) < 1e-2 * abs(float(loss_ref.detach()))
    # with the clamp engaged the hi-plane clamp window adds up to 6e-2 (tests/test_gpu_act_clamp.py)
    bound = 0.15 if conv_clamp in (256.0, None) else 0.2
    assert cos > 0.99 and eg < bound and ee < bound


@pytest.mark.parametrize('cfg,steps,conv_clamp', [pytest.param(c, k, 256.0, id=f'{c}-{k}') for c, k in (('tiny', 3), ('tiny128', 2), ('small', 2))]
                         + [pytest.param('tiny', 3, v, id=f'tiny-3-clamp{v}') for v in (None, 1.0, 0.7)])
@pytest.mark.parametrize('precision', ['fp32_parity', 'bf16'])
def test_augment_loop_with_realism_term(cfg, steps, precision, conv_clamp):
    from oracle import latent_aug as ola
    wl, D, eng = _setup(cfg, precision, conv_clamp=conv_clamp)
    eng.set_latent_bank(wl['W'])
    eng.set_image_bank(wl['X'])
    orc = ola.LatentAugOracle(wl['G'], wl['W'], wl['X'], num_epochs=steps, fused=True, D=D, w_disc=1.0)
    random.seed(0)
    img_ref, w_ref = orc.forward(wl['w0'].clone())
    with torch.no_grad():
        img_ref = wl['G'].synthesis(w_ref, noise_mode='const')
    img, w_aug, losses = eng.augment(wl['w0'], num_steps=steps, lr=0.01, w_latent=1.0, w_pix=1.0, w_disc=1.0,
                                     final_noise_mode='const', return_losses=True)
    eng.debug_check()
    ew, ei = rel_l2(w_aug.cpu(), w_ref[:, 0]), rel_l2(img.cpu(), img_ref)
    l0 = losses[0].cpu()
    print(f'\n[augment+disc {cfg} steps={steps} {precision} conv_clamp={conv_clamp}] rel_w={ew:.3e} rel_img={ei:.3e} '
          f'l_disc ours={float(l0[3]):.6f} oracle={orc.loss_log[0][3]:.6f}')
    assert abs(float(l0[3]) - orc.loss_log[0][3]) <= (1e-2 if precision == 'fp32_parity' else 3e-2) * abs(orc.loss_log[0][3])
    assert ew < TOL[precision] and ei < TOL[precision]
    # the term must actually move w: without it the result differs by far more than the tolerance
    orc0 = ola.LatentAugOracle(wl['G'], wl['W'], wl['X'], num_epochs=steps, fused=True)
    random.seed(0)
    _, w0_ref = orc0.forward(wl['w0'].clone())
    moved = rel_l2(w0_ref[:, 0], w_ref[:, 0])
    print(f'[augment+disc {cfg}] the term moves w by {moved:.3e}')
    assert moved > 2 * ew


def test_realism_term_alone():
    """w_pix = 0, w_latent = 0: the discriminator is the only image-dependent criterion."""
    from oracle import latent_aug as ola
    wl, D, eng = _setup('tiny', 'fp32_parity')
    orc = ola.LatentAugOracle(wl['G'], None, None, num_epochs=3, w_latent=0.0, w_pix=0.0, fused=True, D=D, w_disc=2.0)
    random.seed(0)
    _, w_ref = orc.forward(wl['w0'].clone())
    _, w_aug = eng.augment(wl['w0'], num_steps=3, lr=0.01, w_latent=0.0, w_pix=0.0, w_disc=2.0, final_noise_mode='const')
    ew = rel_l2(w_aug.cpu(), w_ref[:, 0])
    print(f'\n[disc only] rel_w={ew:.3e}')
    assert ew < 1e-3


def test_plugin_with_realism_term():
    """create_augment(opt) with w_disc > 0 in synthetic mode: the reference's default configuration minus lpips."""
    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.options.aug_options import AugOptions
    argv = ['--aug', 'latent', '--synthetic', '--batch_size', '4', '--gpu_ids', '0', '--gpu_ids_aug', '0', '--img_resolution', '32',
            '--synthetic_channels', '2', '--synthetic_bank', '64', '--synthetic_img_bank', '8', '--synthetic_codes', '16',
            '--synthetic_channel_base', '2048', '--synthetic_channel_max', '64', '--precision', 'fp32_parity', '--opt_num_epochs', '3', '--no_log']
    outs = {}
    for w_disc in (0.0, 1.0):
        opt = AugOptions().parse(args={'p_thres': 0.0, 'w_lpips': 0.0, 'w_disc': w_disc, 'init_w': 'inv', 'n_imgs': 0}, argv=argv)
        aug = create_augment(opt)
        names = list(aug.stats_dataset_w.index.keys())[:4]
        img = torch.zeros([4, 1, 32, 32])
        aug.set_input({'A': img, 'B': img, 'A_paths': names, 'B_paths': names})
        aug.forward()
        outs[w_disc] = aug.get_latent_output()['w']
        assert bool(torch.isfinite(aug.get_output()['A']).all())
    import numpy as np
    moved = float(np.linalg.norm(outs[1.0] - outs[0.0]) / np.linalg.norm(outs[0.0]))
    print(f'\n[plugin] realism term moves w by {moved:.3e}')
    assert 1e-3 < moved < 1e-1
