"""The activation clamp with the clamp ENGAGED.  Every convolution epilogue clamps (the reference's
``bias_act(..., clamp=conv_clamp * gain)``), but at the networks' default ``conv_clamp = 256`` no unit of the synthetic
workloads comes near it (99th percentile of |activation| below 5), so the clamp paths only run when ``conv_clamp`` is small.
Here it is 1.0 (exact in bf16, but D's down layers clamp at 1/sqrt(2), which is not) and 0.7 (not exact in bf16), besides
``None`` (no clamp) -- the value of ``--cfg stylegan2`` generators.

What can go wrong.  The backward kernels decide "clamped" from the SAVED output, which is stored in bf16 (hi plane, in
split mode plus a bf16 residual lo plane).  A unit clamped to c is stored as bf16_rn(c) (+ residual), which can be below c;
compared with c itself it reads as unclamped and passes its gradient where the reference's is 0.  The kernels compare with
the clamp as the saved tensor stores it (csrc/act.cuh).  The CPU tests below emulate both rules on the oracle.

CPU tests (no GPU): the clamp is engaged in every generator layer and every clamped D layer of the chosen workloads; which
clamps are bf16-exact; the emulated old rule against the reference (the defect the GPU tolerances must see); and the
tolerance basis -- how far a 1e-6 / 1e-4 relative weight perturbation moves the gradients with the clamp engaged.

Tolerances of the GPU tests, from those measurements (printed by ``test_tolerance_basis_with_the_clamp_engaged``):
  * Images and final ``w`` of loops: the tolerances of tests/test_gpu_parity.py (clamping is 1-Lipschitz, the forward error
    does not grow) -- synthesis 1e-4 / 1e-2, loops 1e-3 (fp32_parity) / 1e-2 (bf16).
  * Per-layer style gradients and d loss / d w of one step, fp32_parity: rel-L2 2e-3.  The split-bf16 forward differs
    from the oracle by ~1e-5 relative; a 1e-4 weight perturbation -- ten times that -- moves the style gradients by at most
    ~4e-4 and d loss / d w by ~3e-4 with the clamp engaged (gate flips of units within the forward error of the clamp or
    of zero).  2e-3 keeps a factor of ~5 above that and sits 10x or more below the emulated defect.
  * Same, bf16: d loss / d w rel-L2 6e-2, per-layer style gradients rel-L2 0.15 and cosine 0.99.  Hi-plane reads keep a
    window of one bf16 step below the clamp where an unclamped unit reads as clamped: emulated on the oracle it alone
    moves d loss / d w by 2-2.5e-2 (``test_emulated_old_rule_is_far_outside_the_gpu_tolerances``), and the 4x4 layer,
    with ~30 % of its units at the clamp, most (measured on a B200: d loss / d w up to 3.4e-2, b4.conv1 up to 9e-2 at
    cosine 0.996).  The old rule at conv_clamp 0.7 gives 0.7 on d loss / d w (emulated) and 1.5-1.8 at cosine 0.55-0.63
    on b4.conv1 (measured): ten times these tolerances.
  * Discriminator: the thresholds of tests/test_gpu_disc.py (fp32_parity input gradient 5e-3, bf16 cosine 0.99 / 0.15).
    The D input gradient is sensitive: a 1e-6 weight perturbation moves it by 0.8-1.7e-3 with the clamp engaged.  D reads
    hi + lo of its saved outputs in fp32_parity, so the fixed rule is exact there to 5e-4 (emulated); measured on a B200
    1.1e-5 .. 3e-3.  The old rule is off by 6e-2 at conv_clamp 1.0 and ~1 at 0.7: ten times the fp32_parity tolerance or
    more.  In bf16 the hi-plane window adds up to 6e-2 (emulated) to the 5-9 % of bf16 rounding alone
    (tests/test_tolerance_basis.py), so with the clamp engaged the bf16 rel-L2 bound is 0.2 (measured 0.09-0.17) and the
    cosine bound stays 0.99; that does not see the old rule's 6e-2 at conv_clamp 1.0, only its ~1.0 at 0.7.
"""
import math
import os
import random
import subprocess
import sys

import pytest
import torch

from conftest import ROOT, rel_l2

TOL = {'fp32_parity': 1e-3, 'bf16': 1e-2}
GRAD_TOL = {'fp32_parity': 2e-3, 'bf16': 6e-2}          # d loss / d w
LAYER_TOL = {'fp32_parity': 2e-3, 'bf16': 0.15}          # per-layer style gradients
GRAD_COS = {'fp32_parity': 0.99999, 'bf16': 0.99}
D_GRAD_TOL_FP32 = 5e-3          # tests/test_gpu_disc.py
CLAMPS = [None, 1.0, 0.7]
SQRT_HALF = math.sqrt(0.5)


# ----------------------------------------------------------------------------------------------------------- oracle side
def set_clamp(G, c):
    """conv_clamp c in every layer of an oracle generator (the attribute is read at each forward)."""
    for m in G.modules():
        if type(m).__name__ in ('SynthLayer', 'ToRGB'):
            m.conv_clamp = c
    return G


def workload(cfg, clamp, batch=None):
    from oracle import synthetic
    wl = synthetic.make_workload(cfg, noise_strength=0.1, batch=batch)
    set_clamp(wl['G'], clamp)
    return wl


def discriminator(c, clamp, mbstd_group_size=4):
    from oracle import sg2_disc
    return sg2_disc.make_discriminator(img_resolution=c['img_resolution'], img_channels=c['img_channels'], channel_base=c['channel_base'],
                                       channel_max=c['channel_max'], conv_clamp=clamp, mbstd_group_size=mbstd_group_size)


def disc_input(c, B):
    return torch.rand([B, c['img_channels'], c['img_resolution'], c['img_resolution']], generator=torch.Generator().manual_seed(11)) * 2 - 1


def disc_input_grad(D, x):
    x = x.clone().requires_grad_(True)
    (torch.nn.functional.softplus(-D(x, c=None)).mean() * 0.7).backward()
    return x.grad


def f32(v):
    return float(torch.tensor(v, dtype=torch.float32))


def bf16(v):
    return float(torch.tensor(v, dtype=torch.float32).bfloat16().float())


def stored_clamp(c, planes):
    """The clamp c as a saved tensor stores it: bf16_rn(c) (hi plane), or hi + bf16_rn(c - hi) summed in fp32 (hi + lo);
    the restatement of csrc/act.cuh::act_saved_clamp."""
    c32 = torch.tensor(c, dtype=torch.float32)
    hi = c32.bfloat16().float()
    return float(hi if planes == 1 else hi + (c32 - hi).bfloat16().float())


class _SavedOutputGate(torch.autograd.Function):
    """clamp(y, -c, c) whose gradient is passed where the STORED output passes |saved| < thr (the kernels' rule)."""

    @staticmethod
    def forward(ctx, y, c, thr, planes):
        out = y.clamp(-c, c)
        hi = out.bfloat16().float()
        ctx.save_for_backward(hi if planes == 1 else hi + (out - hi).bfloat16().float())
        ctx.thr = thr
        return out

    @staticmethod
    def backward(ctx, g):
        (s,) = ctx.saved_tensors
        return g * (s.abs() < ctx.thr).to(g.dtype), None, None, None


def emulate_saved_output_rule(monkeypatch, rule, planes):
    """The oracle's lrelu + clamp layers with the kernels' clamp decision: rule 'old' compares the saved output with c,
    rule 'new' with the clamp as stored.  Linear layers (toRGB) decide on the fp32 pre-clamp value in the kernels too."""
    from oracle import ops
    orig = ops.bias_act

    def bias_act(x, b=None, dim=1, act='linear', alpha=None, gain=None, clamp=None):
        if act == 'linear' or clamp is None or clamp < 0:
            return orig(x, b, dim=dim, act=act, alpha=alpha, gain=gain, clamp=clamp)
        y = orig(x, b, dim=dim, act=act, alpha=alpha, gain=gain, clamp=None)
        thr = f32(clamp) if rule == 'old' else stored_clamp(clamp, planes)
        return _SavedOutputGate.apply(y, f32(clamp), thr, planes)
    monkeypatch.setattr(ops, 'bias_act', bias_act)


def layer_outputs(module, fn):
    """{layer name: |output|} of every clamped lrelu layer of an oracle network during fn()."""
    from oracle import ops
    out, orig = {}, ops.bias_act
    names = {id(m): n for n, m in module.named_modules()}
    stack = []

    def bias_act(x, b=None, dim=1, act='linear', alpha=None, gain=None, clamp=None):
        y = orig(x, b, dim=dim, act=act, alpha=alpha, gain=gain, clamp=clamp)
        if act != 'linear' and clamp is not None and stack:
            out[stack[-1]] = (y.detach().abs(), f32(clamp))
        return y

    def enter(mod, inp):
        stack.append(names[id(mod)])

    def leave(mod, inp, o):
        stack.pop()
    hooks = []
    for m in module.modules():
        if type(m).__name__ in ('SynthLayer', 'Conv2dLayer'):
            hooks += [m.register_forward_pre_hook(enter), m.register_forward_hook(leave)]
    ops.bias_act = bias_act
    try:
        with torch.no_grad():
            fn()
    finally:
        ops.bias_act = orig
        for h in hooks:
            h.remove()
    return out


# chosen workloads: the small oracle configs plus the shapes of the GPU tests that select other kernel variants
G_CASES = {'tiny': 'tiny', 'small': 'small',
           'bn128': dict(img_resolution=64, img_channels=3, channel_base=8192, channel_max=128, batch=4, steps=3, bank=32, img_bank=4),
           'wide1ch': dict(img_resolution=64, img_channels=1, channel_base=16384, channel_max=256, batch=4, steps=2, bank=32, img_bank=4)}
# least fraction of units at the clamp in every generator layer (measured minima 0.8 % / 1.4 %), and in the three clamped
# layers of D's first block (measured minima fromrgb 11 % / 19 %, conv0 5 % / 8 %, conv1 0.05 % / 0.15 %); D's deeper layers
# reach the clamp only sporadically at these values and are not asserted
G_ENGAGED = {1.0: 0.004, 0.7: 0.007}
D_ENGAGED = {'fromrgb': 0.05, 'conv0': 0.025, 'conv1': 2.5e-4}


@pytest.mark.parametrize('clamp', [1.0, 0.7])
@pytest.mark.parametrize('case', list(G_CASES))
def test_clamp_is_engaged_in_every_generator_layer(case, clamp):
    wl = workload(G_CASES[case], clamp)
    G = wl['G']
    ws = wl['w0'].repeat(1, G.num_ws, 1)
    outs = layer_outputs(G, lambda: G.synthesis(ws, noise_mode='const'))
    assert len(outs) == G.num_ws - 1                      # every SynthLayer (all but toRGB of the last block's w)
    fr = {n: float((y >= c).double().mean()) for n, (y, c) in outs.items()}
    print(f'\n[{case} conv_clamp={clamp}] fraction at the clamp per layer: ' + ' '.join(f'{n}={v:.3f}' for n, v in fr.items()))
    low = {n: v for n, v in fr.items() if v < G_ENGAGED[clamp]}
    assert not low, f'clamp not engaged (< {G_ENGAGED[clamp]}) in {low}'
    with torch.no_grad():
        img = G.synthesis(ws, noise_mode='const')
    assert float((img.abs() >= f32(clamp)).double().mean()) > 0.1          # toRGB clamps too


@pytest.mark.parametrize('clamp', [1.0, 0.7])
@pytest.mark.parametrize('cfg', ['tiny', 'tiny128', 'small'])
def test_clamp_is_engaged_in_every_discriminator_layer(cfg, clamp):
    from oracle import synthetic
    c = synthetic.CONFIGS[cfg]
    D = discriminator(c, clamp)
    x = disc_input(c, c['batch'])
    outs = layer_outputs(D, lambda: D(x, c=None))
    fr = {n: float((y >= cl).double().mean()) for n, (y, cl) in outs.items()}
    print(f'\n[D {cfg} conv_clamp={clamp}] fraction at the clamp per layer: ' + ' '.join(f'{n}={v:.4f}' for n, v in fr.items()))
    top = f'b{c["img_resolution"]}.'
    low = {n: v for n, v in fr.items() if n.startswith(top) and v < D_ENGAGED[n[len(top):]]}
    assert len([n for n in fr if n.startswith(top)]) == 3 and 'b4.conv' in fr
    assert not low, f'clamp not engaged in {low} (least fractions {D_ENGAGED})'


def test_bf16_representability_of_the_clamps():
    """Which clamps a bf16-saved output can hold exactly.  256 (G's default) and 1.0 can; D's down layers clamp at
    conv_clamp / sqrt(2) (256 -> 181.019, stored 181.0) and 0.7 cannot -- there the clamped test must use the stored value."""
    assert bf16(256.0) == 256.0 and bf16(1.0) == 1.0
    assert stored_clamp(256.0, 1) == stored_clamp(256.0, 2) == 256.0
    for c in (256 * SQRT_HALF, SQRT_HALF, 0.7, 0.7 * SQRT_HALF):
        assert bf16(c) < f32(c), c                          # hi plane: a clamped unit reads BELOW c under the old rule
    assert bf16(256 * SQRT_HALF) == 181.0
    assert bf16(0.7) == 0.69921875
    # hi + lo: 16 significant bits, within 2^-16 of c on either side (0.7 rounds up, 181.019 down), never the hi plane's value
    for c in (256 * SQRT_HALF, SQRT_HALF, 0.7):
        assert abs(stored_clamp(c, 2) - f32(c)) <= f32(c) * 2 ** -16 and stored_clamp(c, 2) != stored_clamp(c, 1)
    assert stored_clamp(0.7, 2) > f32(0.7) and stored_clamp(256 * SQRT_HALF, 2) < f32(256 * SQRT_HALF)


def _d_grad(cfg, clamp, monkeypatch=None, rule=None, planes=1):
    from oracle import synthetic
    c = synthetic.CONFIGS[cfg]
    D = discriminator(c, clamp)
    x = disc_input(c, c['batch'])
    if rule is None:
        return disc_input_grad(D, x)
    with monkeypatch.context() as m:
        emulate_saved_output_rule(m, rule, planes)
        return disc_input_grad(D, x)


def _g_grads(cfg, clamp, monkeypatch=None, rule=None, planes=1):
    import tools.grad_check as gc
    wl = workload(cfg, clamp)
    if rule is None:
        return gc.oracle_grads(wl, None)
    with monkeypatch.context() as m:
        emulate_saved_output_rule(m, rule, planes)
        return gc.oracle_grads(wl, None)


@pytest.mark.parametrize('clamp', [1.0, 0.7])
@pytest.mark.parametrize('cfg', ['tiny', 'small'])
def test_emulated_old_rule_is_far_outside_the_gpu_tolerances(monkeypatch, cfg, clamp):
    """The old rule (|saved| < c) and the fixed one (|saved| < c as stored) emulated on the oracle against the reference's clamp
    autograd, for the planes each kernel reads: D read the hi plane only before the fix (both precisions) and reads hi + lo
    in fp32_parity now; G reads hi + lo in fp32_parity, hi in bf16.  Where the old rule is wrong the error is at least 10x the
    GPU tolerance that checks it; the fixed rule keeps only the one-bf16-step window below c in hi-plane reads."""
    g_ref = _d_grad(cfg, clamp)
    d = {(rule, planes): rel_l2(_d_grad(cfg, clamp, monkeypatch, rule, planes), g_ref) for rule, planes in (('old', 1), ('new', 1), ('new', 2))}
    ref = _g_grads(cfg, clamp)['grad_w']
    g = {(rule, planes): rel_l2(_g_grads(cfg, clamp, monkeypatch, rule, planes)['grad_w'], ref) for rule in ('old', 'new') for planes in (1, 2)}
    print(f'\n[{cfg} conv_clamp={clamp}] D input gradient vs reference: old rule (hi) {d["old", 1]:.3e}, fixed hi {d["new", 1]:.3e}, '
          f'fixed hi+lo {d["new", 2]:.3e}; G d loss/d w: hi old {g["old", 1]:.3e} fixed {g["new", 1]:.3e}, '
          f'hi+lo old {g["old", 2]:.3e} fixed {g["new", 2]:.3e}')
    # D: conv1 clamps at clamp / sqrt(2), not bf16-exact for either value
    assert d['old', 1] > 10 * D_GRAD_TOL_FP32
    assert d['new', 2] < D_GRAD_TOL_FP32 / 5
    assert d['new', 1] < 0.15 / 2                             # the bf16 thresholds of tests/test_gpu_disc.py
    # G: at 0.7 the hi-plane (bf16) defect is 10x the bf16 gradient and loop tolerances; hi + lo rounds 0.7 up, so the
    # fp32_parity generator was never affected (and neither is any bf16-exact clamp such as 1.0 or 256)
    if clamp == 0.7:
        assert g['old', 1] > 10 * GRAD_TOL['bf16'] and g['old', 1] > 10 * TOL['bf16']
        assert stored_clamp(0.7, 2) > f32(0.7)
    else:
        assert g['old', 1] == g['new', 1]
    assert g['old', 2] == g['new', 2] == 0.0
    assert g['new', 1] < GRAD_TOL['bf16'] / 2


def _perturbed(module, delta, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in module.named_parameters():
            if n.endswith('weight'):
                p.mul_(1.0 + delta * torch.randn(p.shape, generator=g))
    return module


@pytest.mark.parametrize('clamp', [1.0, 0.7])
def test_tolerance_basis_with_the_clamp_engaged(clamp):
    """Gate flips at the clamp boundary: perturb the weights by 1e-6 / 1e-4 (relative) with the clamp engaged and measure how
    far the per-layer style gradients, d loss / d w and the D input gradient move -- the basis of the GPU tolerances."""
    import tools.grad_check as gc
    from oracle import synthetic
    wl = workload('small', clamp)
    ref = gc.oracle_grads(wl, None)
    c = synthetic.CONFIGS['small']
    x = disc_input(c, c['batch'])
    d_ref = disc_input_grad(discriminator(c, clamp), x)
    moved = {}
    for delta in (1e-6, 1e-4):
        wl2 = workload('small', clamp)
        _perturbed(wl2['G'].synthesis, delta, 17)
        got = gc.oracle_grads(wl2, None)
        per_layer = max(rel_l2(got['g_s'][n], ref['g_s'][n]) for n in ref['names'])
        moved[delta] = (per_layer, rel_l2(got['grad_w'], ref['grad_w']),
                        rel_l2(disc_input_grad(_perturbed(discriminator(c, clamp), delta, 19), x), d_ref))
    print(f'\n[conv_clamp={clamp}] weights perturbed by 1e-6 / 1e-4: worst per-layer style gradient {moved[1e-6][0]:.2e} / '
          f'{moved[1e-4][0]:.2e}, d loss/d w {moved[1e-6][1]:.2e} / {moved[1e-4][1]:.2e}, D input gradient '
          f'{moved[1e-6][2]:.2e} / {moved[1e-4][2]:.2e}')
    # at the split-bf16 forward error (~1e-5; geometric mean of the two measurements) the generator's gradients move by a
    # third of the fp32_parity tolerance or less
    at_1e5 = [math.sqrt(moved[1e-6][i] * moved[1e-4][i]) for i in range(3)]
    print(f'interpolated to 1e-5: style {at_1e5[0]:.2e}, d loss/d w {at_1e5[1]:.2e}, D input gradient {at_1e5[2]:.2e}')
    assert at_1e5[0] < GRAD_TOL['fp32_parity'] / 3 and at_1e5[1] < GRAD_TOL['fp32_parity'] / 3
    # the D input gradient is far more sensitive: already a 1e-6 perturbation uses a third of the 5e-3 tolerance or more
    assert moved[1e-6][2] < D_GRAD_TOL_FP32 / 2


# --------------------------------------------------------------------------------------------------------------- GPU side
def _engine(wl, precision, clamp):
    from latentaugment_b200.engine import SynthesisEngine
    G = wl['G']
    return SynthesisEngine(dict(G.state_dict()), img_resolution=G.img_resolution, img_channels=G.img_channels, w_dim=G.w_dim,
                           z_dim=G.z_dim, conv_clamp=clamp, batch=wl['w0'].shape[0], precision=precision)


@pytest.mark.gpu
@pytest.mark.parametrize('seed_stream', [False, True])
@pytest.mark.parametrize('clamp', CLAMPS)
@pytest.mark.parametrize('cfg', ['tiny', 'small', 'wide1ch'])
@pytest.mark.parametrize('precision', ['fp32_parity', 'bf16'])
def test_clamp_style_gradients_per_layer(monkeypatch, cfg, clamp, precision, seed_stream):
    """One optimisation step: the style gradient of every layer and d loss / d w against autograd through the oracle with the
    same conv_clamp (tools/grad_check.py).  LA_SEED_STREAM (read per plan) swaps the bf16 bulk seed pass for the streaming one."""
    import tools.grad_check as gc
    if seed_stream:
        if precision != 'bf16':
            pytest.skip('the bulk seed pass runs in bf16 mode only')
        monkeypatch.setenv('LA_SEED_STREAM', '1')
    wl = workload(G_CASES[cfg], clamp)
    ref = gc.oracle_grads(wl, None)
    eng = _engine(wl, precision, clamp)
    eng.set_latent_bank(wl['W'])
    eng.set_image_bank(wl['X'])
    eng.augment(wl['w0'], num_steps=1, lr=0.01, w_latent=0.0, w_pix=1.0, final_noise_mode='const')
    eng.debug_check()
    B = wl['w0'].shape[0]
    g_s, gw = eng.debug_get('g_s').cpu(), eng.debug_get('grad_w').cpu().reshape(B, -1)
    soff = [int(v) for v in eng.debug_get('soff').cpu().tolist()]
    bad = []
    for nm, off in zip(ref['names'], soff):
        go = ref['g_s'][nm]
        cin = go.shape[1]
        mine = g_s[B * off:B * off + B * cin].reshape(B, cin)
        if nm.endswith('torgb'):
            mine = mine / math.sqrt(cin)            # the engine's toRGB style includes the 1/sqrt(cin) weight gain
        e = rel_l2(mine, go)
        cos = float(torch.nn.functional.cosine_similarity(mine.double().flatten(), go.double().flatten(), dim=0))
        print(f'[{cfg} conv_clamp={clamp} {precision} seed_stream={int(seed_stream)}] {nm:10s} style gradient rel={e:.2e} cos={cos:.6f}')
        if not (e < LAYER_TOL[precision] and cos > GRAD_COS[precision]):
            bad.append(f'{nm} (rel {e:.2e}, cos {cos:.6f})')
    ew = rel_l2(gw, ref['grad_w'])
    print(f'[{cfg} conv_clamp={clamp} {precision}] d loss/d w rel={ew:.2e}')
    assert not bad, f'style gradients off in: {", ".join(bad)}'
    assert ew < GRAD_TOL[precision], ew


@pytest.mark.gpu
@pytest.mark.parametrize('clamp', CLAMPS)
@pytest.mark.parametrize('cfg,steps', [('tiny', 3), ('small', 2)])
@pytest.mark.parametrize('precision', ['fp32_parity', 'bf16'])
def test_clamp_loop_matches_oracle(cfg, steps, clamp, precision):
    """A short loop with the clamp engaged: final w and image against the oracle loop, with the Adam sign-flip count."""
    from oracle import latent_aug as ola
    from test_gpu_bench_shapes import flip_stats
    wl = workload(cfg, clamp)
    G = wl['G']
    eng = _engine(wl, precision, clamp)
    eng.set_latent_bank(wl['W'])
    eng.set_image_bank(wl['X'])
    orc = ola.LatentAugOracle(G, wl['W'], wl['X'], num_epochs=steps, fused=True)
    random.seed(0)
    _, w_ref = orc.forward(wl['w0'].clone())
    with torch.no_grad():
        img_ref = G.synthesis(w_ref, noise_mode='const')
    img, w_aug = eng.augment(wl['w0'], num_steps=steps, lr=0.01, final_noise_mode='const')
    eng.debug_check()
    ew, ei = rel_l2(w_aug.cpu(), w_ref[:, 0]), rel_l2(img.cpu(), img_ref)
    nflip, ew_rest, _ = flip_stats(w_aug.cpu(), w_ref[:, 0])
    print(f'\n[clamp loop {cfg} conv_clamp={clamp} {precision}] rel_w={ew:.3e} rel_img={ei:.3e} sign-flips={nflip}/{w_aug.numel()} '
          f'rel_w(no flips)={ew_rest:.3e}')
    assert ew < TOL[precision] and ei < TOL[precision]


@pytest.mark.gpu
def test_clamp_tests_without_staged_stores_and_tma_fir_passes():
    """LA_NO_STAGED / LA_NO_FIR_TMA are read once per process: the clamp tests in a child process with both set (row-owner
    stores and the sliding-window FIR passes instead of the staged / TMA variants)."""
    env = dict(os.environ, LA_NO_STAGED='1', LA_NO_FIR_TMA='1')
    r = subprocess.run([sys.executable, '-m', 'pytest', '-x', '-q', '-m', 'gpu', '-k', 'clamp and not without_staged',
                        os.path.join(ROOT, 'tests', 'test_gpu_act_clamp.py'), os.path.join(ROOT, 'tests', 'test_gpu_parity.py'),
                        os.path.join(ROOT, 'tests', 'test_gpu_disc.py')],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = (r.stdout or '')[-2000:] + (r.stderr or '')[-1000:]
    assert r.returncode == 0, tail
    assert ' passed' in r.stdout and 'failed' not in r.stdout, tail
