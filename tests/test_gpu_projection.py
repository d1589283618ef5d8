"""GPU parity of the projection into W (DESIGN.md "Projection"): the CUDA path (``SynthesisEngine.set_projection_targets`` /
``projection_loss_grad`` / ``project``, ``invert_dataset``) against ``oracle/projector.py`` run in float64 on the same device.

Tolerances.  The per-sample distance and its image gradient use tests/test_gpu_lpips.py's: loss 1e-4 (fp32_parity) / 2e-2
(bf16); gradient rel-L2 1e-2 + cosine 0.9999 (fp32_parity), cosine 0.95 (bf16) -- gate flips of the ReLU / max-pool stack
bound the gradient, not arithmetic.  Short projections: tests/test_projection_host.py measures the oracle against itself
with the VGG weights perturbed by 1e-6 and 1e-4 (relative) at the `small` shape and 40 steps: the final w moves by 3.3e-3 /
5.1e-3 (relative L2) and the loss log by 3.8e-4 / 3.9e-4 (max relative).  The w error hardly grows with the perturbation:
Adam moves every coordinate by about lr whatever its gradient's size, so a coordinate whose gradient is near zero moves
+lr or -lr on a last-bit difference.  Split-bf16 operands (forward error ~1.5e-5) sit between the two perturbations:
fp32_parity accepts 1e-2 / 1e-3, about 2x the 1e-4 numbers.  bf16 operands (~4e-3) lie beyond them; the gradient error
grows like the square root of the forward error (tests/test_tolerance_basis.py), sqrt(4e-3 / 1e-4) ~ 6x on the part above
the floor: bf16 accepts 3e-2 / 3e-3.
How far the codes drift apart under such a perturbation depends on the shape (at 128 x 128 with one modality the first
B200 runs measured 3e-2 / 1.3e-2 for fp32_parity, with final losses equal to 1e-4).  So each short projection also measures
its own basis in the same run: the float64 oracle against itself with the VGG weights perturbed by the precision's forward
error.  That is 1e-4 for fp32_parity, an upper bound of its 1.5e-5.  For bf16, one rounding is ~4e-3, but the error through
the stack is larger.  By the square-root law, the measured gradient errors give about (0.2 / 0.006)^2 x 1.5e-5 ~ 1.7e-2:
bf16 0.11-0.13 in the targets test here and 0.15-0.2 in tests/test_gpu_lpips.py, split-bf16 5-7e-3.  So bf16 uses 2e-2.
The spread is the largest over three seeded perturbation draws, and the oracle runs cuDNN in its deterministic mode.  So
the bound is the same in every run; only the CUDA result varies, at its own run-to-run level (float atomics).  The CUDA
result must stay within 3x of that spread, or within the fixed tolerances above, whichever is larger.
"""
import pickle
import zipfile

import numpy as np
import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu

TOL = {  # (final w rel-L2, loss-log max relative error)
    'fp32_parity': (1e-2, 1e-3),
    'bf16': (3e-2, 3e-3),
}
FORWARD_ERROR = {'fp32_parity': 1e-4, 'bf16': 2e-2}      # relative VGG weight perturbation of the same-run basis
BASIS_DRAWS = 3
CASES = {   # name -> (res, img_channels, channel_base, channel_max, batch, steps)
    'small': (64, 3, 8192, 128, 4, 40),
    'r128': (128, 1, 8192, 64, 4, 30),
    'r512_pool': (512, 1, 32768, 64, 4, 30),
}


def _setup(res, C, cb, cm, batch, precision, seed_img=5):
    from latentaugment_b200.engine import SynthesisEngine
    from oracle import lpips as olp
    from oracle import sg2
    G = sg2.make_generator(seed=0, noise_strength=0.1, img_resolution=res, img_channels=C, channel_base=cb, channel_max=cm)
    st = olp.random_vgg_state(7, olp.TAPS_SCRIPT)
    eng = SynthesisEngine(dict(G.state_dict()), img_resolution=res, img_channels=C, batch=batch, precision=precision)
    eng.set_lpips(st, taps=olp.TAPS_SCRIPT, crop_size=min(res, 256), per_sample_targets=True)
    return G, st, eng


def _targets(G, batch, seed):
    """Reachable targets: G.synthesis of mapped random z (const noise), so a projection makes real progress."""
    with torch.no_grad():
        w = G.mapping(torch.randn([batch, G.z_dim], generator=torch.Generator().manual_seed(seed)), None)
        return G.synthesis(w, noise_mode='const').clamp(-1, 1)


@pytest.mark.parametrize('precision', ['fp32_parity', 'bf16'])
@pytest.mark.parametrize('shape', [(128, 2, 4), (512, 1, 2)])
def test_per_sample_targets_loss_and_gradient(precision, shape):
    from oracle import projector as opj
    res, C, B = shape
    G, st, eng = _setup(res, C, 8192 if res < 512 else 32768, 64, B, precision)
    x = torch.rand([B, C, res, res], generator=torch.Generator().manual_seed(3)) * 2 - 1
    # targets = the images themselves: distance 0 and no gradient, exactly
    eng.set_projection_targets(x)
    loss, grad = eng.projection_loss_grad(x)
    eng.debug_check()
    # the window is the whole image: a crop origin is refused, not read past the image
    from latentaugment_b200 import _lib
    from latentaugment_b200.engine import _ptr
    with pytest.raises(_lib.LatentAugmentError, match='crop_x = crop_y = 0'):
        _lib.check(eng.lib.la_lpips_loss_grad(eng.handle, _ptr(x.to(eng.device)), res // 2, res // 2, 1.0, 2, _ptr(loss), _ptr(torch.empty_like(grad)),
                                              _ptr(None)))
    assert float(loss.abs().max()) == 0.0 and float(grad.abs().max()) == 0.0
    # permuted targets against oracle autograd (float64, same device)
    perm = torch.arange(B).roll(1)
    eng.set_projection_targets(x[perm])
    loss, grad = eng.projection_loss_grad(x)
    dev = eng.device
    st64 = {k: v.double().to(dev) for k, v in st.items()}
    xr = x.double().to(dev).requires_grad_(True)
    ref = opj.per_sample_distance(st64, xr, opj.target_features(st64, x[perm].double().to(dev)))
    ref.sum().backward()
    el = float(((loss.double() - ref.detach()).abs() / ref.detach().abs()).max())
    eg = rel_l2(grad, xr.grad)
    cos = float(torch.nn.functional.cosine_similarity(grad.flatten().double().cpu(), xr.grad.flatten().cpu(), dim=0))
    print(f'\n[targets {res} C={C} {precision}] loss rel {el:.2e}  grad rel_l2 {eg:.3e} cos {cos:.6f}')
    if precision == 'fp32_parity':
        assert el < 1e-4 and eg < 1e-2 and cos > 0.9999
    else:
        assert el < 2e-2 and cos > 0.95


@pytest.mark.parametrize('precision', ['fp32_parity', 'bf16'])
@pytest.mark.parametrize('case', list(CASES))
def test_short_projection_matches_oracle(precision, case):
    from oracle import projector as opj
    res, C, cb, cm, B, T = CASES[case]
    G, st, eng = _setup(res, C, cb, cm, B, precision)
    y = _targets(G, B, 9)
    eng.set_projection_targets(y)
    noise = torch.randn([T, B, G.w_dim], generator=torch.Generator().manual_seed(4))
    w, losses = eng.project(num_steps=T, w_noise=noise, return_losses=True)
    eng.debug_check()
    w_avg, w_std = eng.w_stats()
    wa_o, ws_o = opj.w_stats(G)
    assert abs(w_std - ws_o) <= 1e-4 * ws_o and np.abs(w_avg - wa_o).max() <= 1e-4 * np.abs(wa_o).max()
    dev = eng.device
    args = (y.double().to(dev), noise.double().to(dev))
    w_ref, l_ref = opj.project(G.to(dev), {k: v.to(dev) for k, v in st.items()}, *args, w_avg=wa_o, w_std=ws_o, num_steps=T)
    delta = FORWARD_ERROR[precision]
    bw = bl = 0.0
    for draw in range(BASIS_DRAWS):       # the largest spread over several seeded perturbations: a fixed, conservative basis
        g = torch.Generator().manual_seed(2 + draw)
        noisy = {k: (v.double() * (1.0 + delta * torch.randn(v.shape, generator=g, dtype=torch.float64)) if k.startswith('features') else v).to(dev)
                 for k, v in st.items()}
        w_p, l_p = opj.project(G, noisy, *args, w_avg=wa_o, w_std=ws_o, num_steps=T)
        bw = max(bw, rel_l2(w_p, w_ref))
        bl = max(bl, float(((l_p - l_ref).abs() / l_ref.abs()).max()))
    G.cpu()
    ew = rel_l2(w, w_ref)
    el = float(((losses.double().cpu() - l_ref).abs() / l_ref.abs()).max())
    print(f'\n[project {case} {precision}] w rel_l2 {ew:.3e} (oracle at {delta:.0e}, max of {BASIS_DRAWS}: {bw:.3e})  loss-log max rel '
          f'{el:.3e} ({bl:.3e})  loss {float(l_ref[0]):.5f} -> {float(l_ref[-1]):.5f}, ours {float(losses[-1]):.5f}')
    assert float(l_ref[-1]) < float(l_ref[0])           # the projection makes progress
    tw, tl = TOL[precision]
    assert ew < max(tw, 3 * bw) and el < max(tl, 3 * bl)


@pytest.mark.parametrize('precision', ['fp32_parity', 'bf16'])
def test_augment_and_project_never_replay_each_others_graph(precision):
    from oracle import synthetic
    res, C, cb, cm, B, _ = CASES['small']
    G, st, eng = _setup(res, C, cb, cm, B, precision)
    wl = synthetic.make_workload('small', noise_strength=0.1, batch=B)
    eng.set_latent_bank(wl['W'])
    eng.set_image_bank(wl['X'])
    kw = dict(num_steps=4, lr=0.01, w_latent=0.5, w_pix=1.0, final_noise_mode='const')
    a_img, a_w = eng.augment(wl['w0'], **kw)
    b_img, b_w = eng.augment(wl['w0'], **kw)
    y = _targets(G, B, 9)
    eng.set_projection_targets(y)
    p_w, p_loss = eng.project(num_steps=5, return_losses=True)       # after augmentations: must not replay their graph
    c_img, c_w = eng.augment(wl['w0'], **kw)                          # after a projection: must not replay its graph
    eng.debug_check()
    r0 = rel_l2(b_w, a_w)
    r1 = rel_l2(c_w, a_w)
    # the same projection on a fresh engine, twice (its run-to-run level)
    _, _, fresh = _setup(res, C, cb, cm, B, precision)
    fresh.set_projection_targets(y)
    f_w, f_loss = fresh.project(num_steps=5, return_losses=True)
    g_w, g_loss = fresh.project(num_steps=5, return_losses=True)
    q0, q1 = rel_l2(g_loss, f_loss), rel_l2(p_loss, f_loss)
    print(f'\n[graphs {precision}] augment run-to-run {r0:.2e}, after a projection {r1:.2e}; projection loss log run-to-run {q0:.2e}, '
          f'after augmentations {q1:.2e}')
    assert r1 <= 10 * r0 + 1e-6 and rel_l2(c_img, a_img) <= 10 * rel_l2(b_img, a_img) + 1e-6
    assert q1 <= 10 * q0 + 1e-6 and rel_l2(p_w, f_w) <= 10 * rel_l2(g_w, f_w) + 1e-6


def test_invert_dataset_end_to_end(tmp_path):
    """G.synthesis(w*) of 8 two-modality images -> image zip -> tools/invert_dataset.py (batch 3: a padded last batch) ->
    create_augment reads the code zip through --interim_dir and runs forward(); the projection loss agrees with the oracle's."""
    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.augments.utils.util_dataset import LatentCodeDataset
    from latentaugment_b200.options.aug_options import AugOptions
    from oracle import projector as opj
    from tools import invert_dataset as cli
    res, C, B, T = 64, 2, 3, 30
    G, st, eng = _setup(res, C, 8192, 64, B, 'fp32_parity')
    y = _targets(G, 8, 21)
    root = tmp_path / 'interim' / 'ds'
    root.mkdir(parents=True)
    names = [f'train/P1/P1_{i:05d}.pickle' for i in (10, 20, 30, 40, 50, 70, 90, 110)]      # slice ids the bank schedules keep
    with zipfile.ZipFile(root / 'imgs.zip', 'w') as z:
        for i, n in enumerate(names):
            img = {m: ((y[i, c] + 1) * 127.5).numpy().astype('float32') for c, m in enumerate(('a', 'b'))}
            z.writestr(n, pickle.dumps(img, pickle.HIGHEST_PROTOCOL))
    gpath, vpath = tmp_path / 'G.pt', tmp_path / 'vgg.pt'
    torch.save(dict(G.state_dict()), gpath)
    torch.save(st, vpath)
    common = ['--interim_dir', str(tmp_path / 'interim'), '--dataset_aug', 'ds', '--dataset_name_aug', 'imgs', '--dataset_w_name', 'codes',
              '--modalities_aug', 'a,b', '--generator_state', str(gpath)]
    cli.main(common + ['--vgg_state', str(vpath), '--batch', str(B), '--num_steps', str(T), '--split', 'train'])
    ds = LatentCodeDataset(str(root / 'codes.zip'), 'train', w_dim=G.w_dim, num_ws=G.num_ws)
    assert ds.fnames == names
    # the first batch again (the targets as the zip round trip gives them), with its loss log, against the oracle; codes
    # agree to run-to-run level (the style gradients are summed with float atomics in no fixed order)
    y = torch.from_numpy(((y + 1) * 127.5).numpy().astype('float32')) / 127.5 - 1
    eng.set_projection_targets(y[:B])
    w, losses = eng.project(num_steps=T, seed=0, return_losses=True)
    assert rel_l2(ds.to_table().lookup(names[:B]).float(), w) < TOL['fp32_parity'][0]
    wa, ws = opj.w_stats(G)
    noise = torch.randn([T, B, G.w_dim], generator=torch.Generator().manual_seed(0))
    dev = eng.device
    _, l_ref = opj.project(G.to(dev), {k: v.to(dev) for k, v in st.items()}, y[:B].double().to(dev), noise.double().to(dev),
                           w_avg=wa, w_std=ws, num_steps=T)
    G.cpu()
    el = abs(float(losses[-1]) - float(l_ref[-1])) / float(l_ref[-1])
    print(f'\n[invert e2e] final loss ours {float(losses[-1]):.6f} oracle {float(l_ref[-1]):.6f} rel {el:.2e}')
    assert el < TOL['fp32_parity'][1]
    argv = ['--aug', 'latent', '--batch_size', '4', '--img_resolution', str(res), '--opt_num_epochs', '2', '--no_log', '--w_lpips', '0',
            '--w_disc', '0'] + common
    opt = AugOptions().parse(args={'p_thres': 0.0, 'init_w': 'inv'}, argv=argv)
    aug = create_augment(opt)
    aug.set_input({'A': torch.zeros(4, 1, res, res), 'B': torch.zeros(4, 1, res, res), 'A_paths': names[:4], 'B_paths': names[:4]})
    aug.forward()
    out = aug.get_output()
    assert out['A'].shape == out['B'].shape == (4, 1, res, res) and bool(torch.isfinite(out['A']).all())
