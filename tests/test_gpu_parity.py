"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same
seeded inputs, and against the reference-generated golden fixtures.

Tolerances (relative L2, written here as the north_star states them):
  * fp32_parity mode (split-bf16 operands, fp32 accumulate): 1e-3 on images and final w
  * bf16 mode: widened to 1e-2 (measured ~2-3e-3, tools/precision_study.py)
  * nearest-code indices: bit-exact
"""
import random

import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu

TOL = {'fp32_parity': 1e-3, 'bf16': 1e-2}


def _engine(wl, precision, batch=None, conv_clamp=256.0):
    from latentaugment_b200.engine import SynthesisEngine
    G = wl['G']
    return SynthesisEngine(dict(G.state_dict()), img_resolution=G.img_resolution, img_channels=G.img_channels,
                           w_dim=G.w_dim, z_dim=G.z_dim, conv_clamp=conv_clamp, batch=batch or wl['w0'].shape[0], precision=precision)


def _workload(cfg, noise_strength=0.1, conv_clamp=256.0):
    from oracle import synthetic
    return synthetic.make_workload(cfg, noise_strength=noise_strength, conv_clamp=conv_clamp)


def with_clamps(cases, clamps=(None, 1.0, 0.7)):
    """Parameters (case, conv_clamp): every case at the networks' default 256 under its plain id, then the clamp off (None)
    and engaged (1.0 is bf16-exact, 0.7 is not; tests/test_gpu_act_clamp.py) -- ids ``<case>-clamp<value>``."""
    out = [pytest.param(c, 256.0, id=str(c)) for c in cases]
    return out + [pytest.param(c, v, id=f'{c}-clamp{v}') for v in clamps for c in cases]


@pytest.mark.parametrize('cfg,conv_clamp', with_clamps(['tiny', 'tiny128', 'small'])[:3] + with_clamps(['tiny'])[1:])
@pytest.mark.parametrize('precision', ['fp32_parity', 'bf16'])
def test_synthesis_matches_oracle(cfg, precision, conv_clamp):
    wl = _workload(cfg, conv_clamp=conv_clamp)
    G = wl['G']
    eng = _engine(wl, precision, conv_clamp=conv_clamp)
    ws = wl['w0'].repeat(1, G.num_ws, 1)
    with torch.no_grad():
        ref_const = G.synthesis(ws, noise_mode='const')
        ref_none = G.synthesis(ws, noise_mode='none')
    out_const = eng.synthesis(ws, noise_mode='const').cpu()
    out_none = eng.synthesis(ws, noise_mode='none').cpu()
    eng.debug_check()
    e1, e2 = rel_l2(out_const, ref_const), rel_l2(out_none, ref_none)
    print(f'\n[synthesis {cfg} {precision} conv_clamp={conv_clamp}] rel_l2 const={e1:.3e} none={e2:.3e}')
    tol = 1e-4 if precision == 'fp32_parity' else 1e-2
    assert e1 < tol and e2 < tol
    # distinct ws rows per layer (general G.synthesis(ws) call)
    ws2 = ws + 0.05 * torch.randn(ws.shape, generator=torch.Generator().manual_seed(9))
    with torch.no_grad():
        ref2 = G.synthesis(ws2, noise_mode='const')
    e3 = rel_l2(eng.synthesis(ws2, noise_mode='const').cpu(), ref2)
    print(f'[synthesis {cfg} {precision}] per-layer ws rel_l2={e3:.3e}')
    assert e3 < tol


@pytest.mark.parametrize('cfg', ['tiny', 'tiny128'])
def test_tensor_core_path_matches_simt_twin(cfg):
    """tcgen05 tap-GEMM vs its SIMT twin (same epilogue code, brute-force accumulation)."""
    wl = _workload(cfg)
    G = wl['G']
    eng = _engine(wl, 'fp32_parity')
    ws = wl['w0'].repeat(1, G.num_ws, 1)
    a = eng.synthesis(ws, noise_mode='const').cpu()
    eng.debug_set_simt(1)
    b = eng.synthesis(ws, noise_mode='const').cpu()
    eng.debug_set_simt(0)
    e = rel_l2(a, b)
    print(f'\n[tc vs simt {cfg}] rel_l2={e:.3e}')
    assert e < 2e-5


def test_random_noise_synthesis_matches_oracle():
    wl = _workload('tiny')
    G = wl['G']
    eng = _engine(wl, 'fp32_parity')
    ws = wl['w0'].repeat(1, G.num_ws, 1)
    torch.manual_seed(77)
    with torch.no_grad():
        ref = G.synthesis(ws, noise_mode='random')
    torch.manual_seed(77)       # same draws, same layer order (conv0, conv1 per block)
    noise = [torch.randn([ws.shape[0], 1, r, r]) for r in eng.conv_res]
    out = eng.synthesis(ws, noise_mode='random', noise=noise).cpu()
    e = rel_l2(out, ref)
    print(f'\n[random noise] rel_l2={e:.3e}')
    assert e < 1e-4


@pytest.mark.parametrize('cfg,steps', [('tiny', 3), ('tiny128', 2), ('small', 2), ('tiny', 10)])
@pytest.mark.parametrize('precision', ['fp32_parity', 'bf16'])
def test_augment_loop_matches_oracle(cfg, steps, precision):
    from oracle import latent_aug as ola
    wl = _workload(cfg)
    G = wl['G']
    eng = _engine(wl, precision)
    eng.set_latent_bank(wl['W'])
    eng.set_image_bank(wl['X'])
    orc = ola.LatentAugOracle(G, wl['W'], wl['X'], num_epochs=steps, fused=True)
    random.seed(0)
    torch.manual_seed(1234)
    img_ref, w_ref = orc.forward(wl['w0'].clone())
    torch.manual_seed(1234)
    noise = [torch.randn([wl['w0'].shape[0], 1, r, r]) for r in eng.conv_res]
    img, w_aug, losses = eng.augment(wl['w0'], num_steps=steps, lr=0.01, w_latent=1.0, w_pix=1.0,
                                     final_noise_mode='random', final_noise=noise, return_losses=True)
    eng.debug_check()
    ew, ei = rel_l2(w_aug.cpu(), w_ref[:, 0]), rel_l2(img.cpu(), img_ref)
    l0 = losses[0].cpu()
    print(f'\n[augment {cfg} steps={steps} {precision}] rel_w={ew:.3e} rel_img={ei:.3e} '
          f'loss0 ours=({l0[0]:.6f},{l0[1]:.6f}) oracle=({orc.loss_log[0][0]:.6f},{orc.loss_log[0][1]:.6f})')
    assert abs(float(l0[0]) - orc.loss_log[0][0]) <= 1e-4 * abs(orc.loss_log[0][0])
    assert abs(float(l0[1]) - orc.loss_log[0][1]) <= (1e-3 if precision == 'fp32_parity' else 2e-2) * abs(orc.loss_log[0][1])
    assert ew < TOL[precision] and ei < TOL[precision]


@pytest.mark.parametrize('name', ['loop_tiny.pt', 'loop_tiny_soft.pt', 'loop_tiny128.pt', 'loop_small.pt', 'loop_c1.pt'])
def test_augment_loop_matches_reference_golden(golden, name):
    """Against outputs of the REFERENCE's own LatentAug.forward (tests/golden, oracle/make_golden.py)."""
    g = golden(name)
    wl = _workload(g['config'], noise_strength=g['noise_strength'])
    eng = _engine(wl, 'fp32_parity')
    eng.set_latent_bank(wl['W'])
    eng.set_image_bank(wl['X'])
    G = wl['G']
    ws0 = wl['w0'].repeat(1, G.num_ws, 1)
    e0 = rel_l2(eng.synthesis(ws0, noise_mode='const').cpu(), g['img0_const'])
    torch.manual_seed(1234)
    noise = [torch.randn([wl['w0'].shape[0], 1, r, r]) for r in eng.conv_res]
    img, w_aug, losses = eng.augment(wl['w0'], num_steps=g['steps'], lr=0.01, w_latent=g['w_latent'], w_pix=g['w_pix'],
                                     soft_aug=g['soft_aug'], alpha=g['alpha'], final_noise_mode='random', final_noise=noise,
                                     return_losses=True)
    ew, ei = rel_l2(w_aug.cpu(), g['w_aug']), rel_l2(img.cpu(), g['img'])
    print(f'\n[golden {name}] img0={e0:.3e} rel_w={ew:.3e} rel_img={ei:.3e}')
    assert e0 < 1e-4
    assert abs(float(losses[0, 0]) - g['loss_latent0']) <= 1e-4 * abs(g['loss_latent0'])
    assert abs(float(losses[0, 1]) - g['loss_pix0']) <= 1e-3 * abs(g['loss_pix0'])
    assert ew < 1e-3 and ei < 1e-3


def test_latent_only_and_zero_steps():
    """w_pix = 0 skips synthesis in the loop; num_steps = 0 is the rand_aug configuration."""
    from oracle import latent_aug as ola
    wl = _workload('tiny', noise_strength=0.0)
    G = wl['G']
    eng = _engine(wl, 'fp32_parity')
    eng.set_latent_bank(wl['W'])
    orc = ola.LatentAugOracle(G, wl['W'], None, num_epochs=4, w_pix=0.0)
    img_ref, w_ref = orc.forward(wl['w0'].clone())
    img, w_aug = eng.augment(wl['w0'], num_steps=4, w_pix=0.0, final_noise_mode='const')
    assert rel_l2(w_aug.cpu(), w_ref[:, 0]) < 1e-5
    assert rel_l2(img.cpu(), img_ref) < 1e-4
    img0, w0 = eng.augment(wl['w0'], num_steps=0, w_pix=0.0, final_noise_mode='const')
    assert torch.equal(w0.cpu(), wl['w0'][:, 0])


def test_mapping_matches_oracle():
    wl = _workload('tiny')
    G = wl['G']
    eng = _engine(wl, 'fp32_parity')
    z = torch.randn([3, G.z_dim], generator=torch.Generator().manual_seed(4))
    G.mapping.w_avg.copy_(torch.randn([G.w_dim], generator=torch.Generator().manual_seed(5)) * 0.1)
    eng2 = _engine(wl, 'fp32_parity')
    for psi in (1.0, 0.7):
        with torch.no_grad():
            ref = G.mapping(z, None, truncation_psi=psi)
        out = eng2.mapping(z, truncation_psi=psi).cpu()
        assert out.shape == ref.shape
        e = rel_l2(out, ref)
        print(f'\n[mapping psi={psi}] rel_l2={e:.3e}')
        assert e < 1e-5
    del eng


@pytest.mark.parametrize('shape', [(32, 4096, 7168), (5, 300, 512), (130, 1000, 512)])
def test_nearest_codes_bit_exact(shape):
    from latentaugment_b200.engine import LatentBank, merge_topk, pairwise_sqdist
    from oracle import latent_aug as ola
    n, m, K = shape
    gen = torch.Generator().manual_seed(11)
    Y = torch.randn([m, K], generator=gen)
    X = Y[torch.randint(0, m, [n], generator=gen)] + 0.3 * torch.randn([n, K], generator=gen)
    d_ref, i_ref = ola.nearest_codes(X, Y, k=4)
    D = pairwise_sqdist(X.cuda(), Y.cuda()).cpu()
    D_ref = ola.l2_loss_vectorized(X, Y, compute_mean=False)
    assert D.shape == D_ref.shape == (m, n)
    torch.testing.assert_close(D, D_ref, rtol=1e-5, atol=1e-3)
    bank = LatentBank(Y.cuda())
    dist, idx = bank.nearest(X.cuda(), k=4)
    assert torch.equal(idx.cpu(), i_ref), (idx.cpu()[:4], i_ref[:4])
    torch.testing.assert_close(dist.cpu(), d_ref, rtol=1e-5, atol=1e-3)
    # sharded bank + merge == whole bank
    half = m // 2
    parts = [LatentBank(Y[:half].cuda(), 0).nearest(X.cuda(), k=4), LatentBank(Y[half:].cuda(), half).nearest(X.cuda(), k=4)]
    md, mi = merge_topk(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
    assert torch.equal(mi.cpu(), i_ref)


def test_plugin_api_end_to_end():
    """create_augment(opt) -> set_input / forward / get_output / get_latent_* (reference README.md:66-86 usage),
    synthetic mode; the result must equal the oracle loop started from the same inverted codes."""
    import random as pyrandom

    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.options.aug_options import AugOptions
    from oracle import latent_aug as ola
    from oracle import sg2
    argv = ['--aug', 'latent', '--synthetic', '--batch_size', '4', '--img_resolution', '32', '--synthetic_channels', '2',
            '--synthetic_channel_base', '2048', '--synthetic_channel_max', '64', '--synthetic_bank', '64', '--synthetic_img_bank', '8',
            '--synthetic_codes', '16', '--opt_num_epochs', '3', '--no_log']
    opt = AugOptions().parse(args={'p_thres': 0.0, 'w_lpips': 0.0, 'w_disc': 0.0, 'init_w': 'inv'}, argv=argv)
    aug = create_augment(opt)
    names = list(aug.stats_dataset_w.index)[:4]
    data = {'A': torch.zeros(4, 1, 32, 32), 'B': torch.zeros(4, 1, 32, 32), 'A_paths': names, 'B_paths': names}
    aug.set_input(data)
    pyrandom.seed(3)
    aug.forward()
    out = aug.get_output()
    assert out['A'].shape == (4, 1, 32, 32) and out['B'].shape == (4, 1, 32, 32) and out['A_paths'] == names
    assert not out['A'].is_cuda and len(aug.stats_time) == 1 and aug.num_ws == 8
    w_in, w_out = aug.get_latent_input()['w'], aug.get_latent_output()['w']
    assert w_in.shape == (4, 512) and w_out.shape == (4, 512)
    # oracle over the same generator parameters / banks / init codes
    core = aug.latent_aug.module
    G = sg2.Generator(img_resolution=32, img_channels=2, channel_base=2048, channel_max=64).eval().requires_grad_(False)
    from latentaugment_b200.utils import synthetic
    G.load_state_dict(synthetic.random_generator_state(img_resolution=32, img_channels=2, channel_base=2048, channel_max=64))
    orc = ola.LatentAugOracle(G, core.W.cpu(), core.X.cpu(), num_epochs=3)
    img_ref, w_ref = orc.forward(torch.from_numpy(w_in).reshape(4, 1, 512))
    assert rel_l2(torch.from_numpy(w_out), w_ref[:, 0]) < 1e-3
    ref = torch.cat([img_ref[:, 0:1], img_ref[:, 1:2]], 1)
    got = torch.cat([out['A'], out['B']], 1)
    e = rel_l2(got, ref)
    print(f'\n[plugin api] rel_img={e:.3e}')
    assert e < 1e-3          # noise_strength = 0 in synthetic mode, so the random final noise is immaterial
    # p_thres = 1 (CLI default): never augments, passes the real pair through (reference latent_aug.py:241,268)
    aug.p_thres = 1.0
    aug.forward()
    assert torch.equal(aug.get_output()['A'], data['A'])


@pytest.mark.parametrize('split_min_res', ['8', '100000'])
@pytest.mark.parametrize('precision,conv_clamp', with_clamps(['fp32_parity', 'bf16']))
def test_both_upconv_formulations(monkeypatch, split_min_res, precision, conv_clamp):
    """x2 layers as transposed-conv GEMM + FIR pass (split) and with the FIR folded into 36 taps: both
    must match the oracle, at every resolution (LA_UPCONV_SPLIT_MIN_RES picks per layer)."""
    from oracle import latent_aug as ola
    monkeypatch.setenv('LA_UPCONV_SPLIT_MIN_RES', split_min_res)
    for cfg in ('tiny', 'small'):
        wl = _workload(cfg, conv_clamp=conv_clamp)
        G = wl['G']
        eng = _engine(wl, precision, conv_clamp=conv_clamp)
        eng.set_latent_bank(wl['W'])
        eng.set_image_bank(wl['X'])
        ws = wl['w0'].repeat(1, G.num_ws, 1)
        with torch.no_grad():
            ref = G.synthesis(ws, noise_mode='const')
        e0 = rel_l2(eng.synthesis(ws, noise_mode='const').cpu(), ref)
        orc = ola.LatentAugOracle(G, wl['W'], wl['X'], num_epochs=2)
        random.seed(0)
        img_ref, w_ref = orc.forward(wl['w0'].clone())
        with torch.no_grad():
            img_ref = G.synthesis(w_ref, noise_mode='const')
        img, w_aug = eng.augment(wl['w0'], num_steps=2, final_noise_mode='const')
        eng.debug_check()
        ew, ei = rel_l2(w_aug.cpu(), w_ref[:, 0]), rel_l2(img.cpu(), img_ref)
        print(f'\n[upconv split_min_res={split_min_res} {cfg} {precision} conv_clamp={conv_clamp}] synth={e0:.3e} rel_w={ew:.3e} rel_img={ei:.3e}')
        assert e0 < (1e-4 if precision == 'fp32_parity' else 1e-2)
        assert ew < TOL[precision] and ei < TOL[precision]
        # tensor-core path against the SIMT twin on this formulation
        a = eng.synthesis(ws, noise_mode='const').cpu()
        eng.debug_set_simt(1)
        b = eng.synthesis(ws, noise_mode='const').cpu()
        eng.debug_set_simt(0)
        assert rel_l2(a, b) < (2e-5 if precision == 'fp32_parity' else 5e-3)   # bf16: roundings of intermediates differ


@pytest.mark.parametrize('batch', [1, 3, 5])
@pytest.mark.parametrize('precision', ['fp32_parity', 'bf16'])
def test_ragged_batches(batch, precision):
    """Batch sizes that leave partial M tiles at every resolution (8 / 2 / 1 samples per tile) and odd tile pairs."""
    from oracle import latent_aug as ola
    from oracle import synthetic
    wl = synthetic.make_workload('tiny', noise_strength=0.1, batch=batch)
    G = wl['G']
    eng = _engine(wl, precision, batch=batch)
    eng.set_latent_bank(wl['W'])
    eng.set_image_bank(wl['X'])
    orc = ola.LatentAugOracle(G, wl['W'], wl['X'], num_epochs=2, fused=True)
    random.seed(0)
    _, w_ref = orc.forward(wl['w0'].clone())
    with torch.no_grad():
        img_ref = G.synthesis(w_ref, noise_mode='const')
    img, w_aug = eng.augment(wl['w0'], num_steps=2, final_noise_mode='const')
    eng.debug_check()
    ew, ei = rel_l2(w_aug.cpu(), w_ref[:, 0]), rel_l2(img.cpu(), img_ref)
    print(f'\n[ragged batch={batch} {precision}] rel_w={ew:.3e} rel_img={ei:.3e}')
    assert ew < TOL[precision] and ei < TOL[precision]


def test_single_channel_wide_generator():
    """1-channel images and 256-wide layers at 64^2 (BN = 256 path, TMA FIR passes, bulk seed kernel) against the oracle."""
    _single_channel_wide(256.0)


@pytest.mark.parametrize('conv_clamp', [None, 1.0, 0.7])
def test_single_channel_wide_generator_clamped(conv_clamp):
    _single_channel_wide(conv_clamp)


def _single_channel_wide(conv_clamp):
    from oracle import latent_aug as ola
    from oracle import synthetic
    cfg = dict(img_resolution=64, img_channels=1, channel_base=16384, channel_max=256, batch=4, steps=2, bank=32, img_bank=4)
    wl = synthetic.make_workload(cfg, noise_strength=0.1, conv_clamp=conv_clamp)
    G = wl['G']
    for precision in ('fp32_parity', 'bf16'):
        eng = _engine(wl, precision, conv_clamp=conv_clamp)
        eng.set_latent_bank(wl['W'])
        eng.set_image_bank(wl['X'])
        orc = ola.LatentAugOracle(G, wl['W'], wl['X'], num_epochs=2, fused=True)
        random.seed(0)
        _, w_ref = orc.forward(wl['w0'].clone())
        with torch.no_grad():
            img_ref = G.synthesis(w_ref, noise_mode='const')
        img, w_aug = eng.augment(wl['w0'], num_steps=2, final_noise_mode='const')
        eng.debug_check()
        ew, ei = rel_l2(w_aug.cpu(), w_ref[:, 0]), rel_l2(img.cpu(), img_ref)
        print(f'\n[1-ch wide {precision} conv_clamp={conv_clamp}] rel_w={ew:.3e} rel_img={ei:.3e}')
        assert ew < TOL[precision] and ei < TOL[precision]


def test_in_process_two_gpus():
    """The reference's DataParallel form (--gpu_ids_aug 0,1; util_latent_aug.py:20-33): one resident engine per GPU id in
    ONE process.  Per-device kernel attributes / workspaces must be set up on every device (ADVICE r1)."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs in one process')
    import random as pyrandom

    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.options.aug_options import AugOptions
    argv = ['--aug', 'latent', '--synthetic', '--batch_size', '4', '--img_resolution', '64', '--synthetic_channels', '2',
            '--synthetic_channel_base', '8192', '--synthetic_channel_max', '128', '--synthetic_bank', '64', '--synthetic_img_bank', '8',
            '--synthetic_codes', '16', '--opt_num_epochs', '2', '--no_log']
    outs = []
    for ids in ('0', '0,1'):
        opt = AugOptions().parse(args={'p_thres': 0.0, 'w_lpips': 0.0, 'w_disc': 0.0, 'init_w': 'inv'}, argv=argv + ['--gpu_ids_aug', ids])
        aug = create_augment(opt)
        names = list(aug.stats_dataset_w.index)[:4]
        aug.set_input({'A': torch.zeros(4, 1, 64, 64), 'B': torch.zeros(4, 1, 64, 64), 'A_paths': names, 'B_paths': names})
        pyrandom.seed(3)
        aug.forward()
        outs.append((aug.get_output()['A'].clone(), aug.get_latent_output()['w'].copy()))
        for e in aug.latent_aug.module.engines:
            e.debug_check()
    # per-replica loss normalisers differ (n = batch / world, as under DataParallel), so the two runs agree only loosely;
    # what is asserted is that the second device ran at all and produced finite, close results
    assert torch.isfinite(outs[1][0]).all()
    assert rel_l2(outs[1][0], outs[0][0]) < 0.2


@pytest.mark.parametrize('kind', ['cluster_in_one_tile', 'all_codes_nearly_equal', 'exact_ties'])
def test_nearest_codes_exact_on_adversarial_banks(kind):
    """Banks built to defeat the bf16 candidate pass: many near-identical codes inside the same 32-code chunks (the chunk's
    two-entry candidate list overflows -> exhaustive rescan of the chunk), a bank whose codes differ by less than the bf16
    rounding (every chunk overflows -> whole-shard scan), and exact duplicates (ties go to the lowest index)."""
    from latentaugment_b200.engine import LatentBank
    from oracle import latent_aug as ola
    gen = torch.Generator().manual_seed(5)
    K, m, n = 512, 1500, 24
    Y = torch.randn([m, K], generator=gen)
    X = torch.randn([n, K], generator=gen)
    if kind == 'cluster_in_one_tile':
        Y[300:340] = X[3] + 1e-3 * torch.randn([40, K], generator=gen)        # 40 codes within bf16 noise of query 3, groups 2 / 3 of tile 1
        Y[1290:1300] = X[7] + 1e-4 * torch.randn([10, K], generator=gen)
    elif kind == 'all_codes_nearly_equal':
        Y = Y[:1].repeat(m, 1) + 1e-3 * torch.randn([m, K], generator=gen)
    else:
        Y[500:520] = Y[100]                                                    # 21 identical codes
        X[0] = Y[100] + 0.01 * torch.randn([K], generator=gen)
    # The index contract: order by D = (fl32(|y|^2) + fl32(|x|^2)) - 2 fl32(<x, y>) with the three reductions accumulated in
    # fp64 and rounded once (the reference's association, util_latent_aug.py:336-340), ties to the lowest index.  Against the
    # reference's own fp32 einsum the indices agree wherever its distances are separated by more than its rounding noise
    # (asserted on the random shapes of test_nearest_codes_bit_exact); codes built to lie within that noise need the
    # exactly-defined distance as the checker.
    yy = Y.double().square().sum(1).float()
    xx = X.double().square().sum(1).float()
    yx = (X.double() @ Y.double().t()).float()
    D = (yy[None, :] + xx[:, None]) - 2 * yx                                   # [n, m]
    d_ref, i_ref = torch.sort(D, dim=1, stable=True)
    d_ref, i_ref = d_ref[:, :8].contiguous(), i_ref[:, :8].contiguous()
    dist, idx = LatentBank(Y.cuda()).nearest(X.cuda(), k=8)
    same = torch.equal(idx.cpu(), i_ref)
    d_o, i_o = ola.nearest_codes(X, Y, k=8)
    print(f'\n[nearest {kind}] indices equal to the exactly-defined order: {same}; equal to the fp32-einsum oracle in '
          f'{int((idx.cpu() == i_o).sum())}/{i_o.numel()} slots')
    assert same
    assert torch.equal(dist.cpu(), d_ref)
    if kind == 'exact_ties':
        assert idx[0, 0].item() == 100 and idx[0, 1].item() == 500             # duplicates: lowest index first


def test_micro_batches_and_lookahead_loop_match_plain_calls():
    """--micro_batches 2 (two concurrent half-batch engines, term weights rescaled to the replica's normaliser) and the
    look-ahead caller loop iterate() give the same images as the plain set_input / forward / get_output sequence."""
    import random as pyrandom

    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.options.aug_options import AugOptions
    argv = ['--aug', 'latent', '--synthetic', '--batch_size', '4', '--img_resolution', '64', '--synthetic_channels', '2',
            '--synthetic_channel_base', '8192', '--synthetic_channel_max', '128', '--synthetic_bank', '64', '--synthetic_img_bank', '8',
            '--synthetic_codes', '16', '--opt_num_epochs', '3', '--no_log']
    args = {'p_thres': 0.0, 'w_lpips': 0.0, 'w_disc': 0.0, 'init_w': 'inv'}
    plain = create_augment(AugOptions().parse(args=dict(args), argv=argv))
    micro = create_augment(AugOptions().parse(args=dict(args), argv=argv + ['--micro_batches', '2']))
    names = list(plain.stats_dataset_w.index)
    batches = [{'A': torch.zeros(4, 1, 64, 64), 'B': torch.zeros(4, 1, 64, 64), 'A_paths': names[4 * i:4 * i + 4], 'B_paths': names[4 * i:4 * i + 4]}
               for i in range(3)]
    ref = []
    for data in batches:
        plain.set_input(data)
        pyrandom.seed(1)
        plain.forward()
        ref.append(plain.get_output()['A'].clone())
    # micro-batches
    for data, r in zip(batches, ref):
        micro.set_input(data)
        pyrandom.seed(1)
        micro.forward()
        e = rel_l2(micro.get_output()['A'], r)
        print(f'\n[micro-batches] rel_img={e:.3e}')
        assert e < 1e-3
    # look-ahead loop: same values, outputs stay valid until the next-but-one batch
    pyrandom.seed(1)
    got = []
    for data, out in plain.iterate(iter(batches)):
        got.append((data['A_paths'], out['A'].clone(), out['A_paths']))
    assert len(got) == 3
    for (paths, img, out_paths), data, r in zip(got, batches, ref):
        assert paths == data['A_paths'] == out_paths
        assert rel_l2(img, r) < 1e-5


@pytest.mark.parametrize('precision,conv_clamp', with_clamps(['fp32_parity', 'bf16']))
def test_bn128_layers_match_oracle(precision, conv_clamp):
    """128-channel layers on a grid with more than 74 M tiles select the BN = 128 kernels (two M tiles per unit sharing each
    weight tile; CTA-pair four-tile work items in the forward conv) -- the variant the 256x256 layers of config C2 run.
    64x64 with batch 4 reaches it at a size the oracle finishes in seconds."""
    from oracle import latent_aug as ola
    from oracle import synthetic
    cfg = dict(img_resolution=64, img_channels=3, channel_base=8192, channel_max=128, batch=4, steps=3, bank=32, img_bank=4)
    wl = synthetic.make_workload(cfg, noise_strength=0.1, conv_clamp=conv_clamp)
    G = wl['G']
    eng = _engine(wl, precision, conv_clamp=conv_clamp)
    eng.set_latent_bank(wl['W'])
    eng.set_image_bank(wl['X'])
    orc = ola.LatentAugOracle(G, wl['W'], wl['X'], num_epochs=3, fused=True)
    random.seed(0)
    _, w_ref = orc.forward(wl['w0'].clone())
    with torch.no_grad():
        img_ref = G.synthesis(w_ref, noise_mode='const')
    img, w_aug = eng.augment(wl['w0'], num_steps=3, final_noise_mode='const')
    eng.debug_check()
    d = (w_aug.cpu() - w_ref[:, 0]).abs()
    ew, ei = rel_l2(w_aug.cpu(), w_ref[:, 0]), rel_l2(img.cpu(), img_ref)
    print(f'\n[BN=128 layers {precision} conv_clamp={conv_clamp}] rel_w={ew:.3e} rel_img={ei:.3e} components off by > lr: {int((d > 0.01).sum())}/{d.numel()}')
    assert ew < TOL[precision] and ei < TOL[precision]
