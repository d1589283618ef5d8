"""VGG16 detector on the GPU (csrc/detector.cu, DESIGN.md §13) against the fp32 oracle (oracle/detector.py), its isolation
from an engine's perceptual term and projection, and precision / recall straight from images.

Tolerance basis (tests/test_detector_host.py::test_tolerance_basis measures it on the oracle, 64^2 inputs, seeded state 7):
perturbing every weight by a relative 2^-9 (one bf16 rounding) moves the fc7 features by a relative L2 of BASIS_BF16; by
2^-17 (what the split hi / lo operands keep) by BASIS_SPLIT.  The native paths round the input and the fifteen stored
activations (conv outputs, fc6) the same way besides the weights, so each tolerance is a multiple of its basis: 5x in bf16,
20x in fp32_parity (measured on one B200: 2.5e-4 at every input size, 11x the basis)."""
import pytest
import torch

from oracle import detector as od
from oracle import precision_recall as opr

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'

BASIS_BF16 = 6.0e-3
BASIS_SPLIT = 2.3e-5
TOL = {'bf16': 5 * BASIS_BF16, 'fp32_parity': 20 * BASIS_SPLIT}


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm())


def _oracle(state, img, modality):
    cudnn, mm = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            return od.detector_features(state, img.to(DEV), modality)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = cudnn, mm


def _images(n, C, res, seed):
    """Smooth structure plus noise, a few pixels beyond [-1, 1] (the quantiser clamps them)."""
    g = torch.Generator().manual_seed(seed)
    low = torch.nn.functional.interpolate(torch.randn([n, C, 8, 8], generator=g), size=(res, res), mode='bilinear', align_corners=False)
    return (0.6 * low + 0.3 * torch.randn([n, C, res, res], generator=g)).clamp(-1.1, 1.1)


@pytest.fixture(scope='module')
def state():
    return od.random_detector_state(7)


CASES = {   # name -> (res, img_channels, n, detector batch)
    'r64_ragged': (64, 1, 5, 4),
    'r128_2mod': (128, 2, 3, 8),
    'r256_n1': (256, 1, 1, 4),
    'r512_2mod': (512, 2, 3, 2),
}


@pytest.mark.parametrize('precision', ['bf16', 'fp32_parity'])
@pytest.mark.parametrize('case', list(CASES))
def test_features_match_oracle(state, precision, case):
    from latentaugment_b200.engine import FeatureDetector
    res, C, n, batch = CASES[case]
    det = FeatureDetector(state, batch=batch, precision=precision)
    img = _images(n, C, res, seed=res + C)
    for c in range(C):
        got = det.features(img, modality=c)
        assert got.shape == (n, 4096) and got.dtype == torch.float32 and got.device.type == 'cuda'
        ref = _oracle(state, img, c)
        err = rel(got, ref)
        assert err < TOL[precision], (case, c, err)
        per_image = [rel(got[i], ref[i]) for i in range(n)]
        assert max(per_image) < 2 * TOL[precision], per_image


def test_rejections(state):
    import ctypes as C

    from latentaugment_b200 import _lib
    from latentaugment_b200.engine import FeatureDetector
    det = FeatureDetector(state, batch=4)
    img = torch.zeros([4, 2, 64, 64], device=DEV)
    out = torch.empty([4, 4096], device=DEV)
    p = lambda t: C.c_void_p(t.data_ptr())          # noqa: E731
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for n, c, res, mod in ((0, 2, 64, 0), (5, 2, 64, 0), (4, 2, 64, 2), (4, 2, 64, -1), (4, 2, 15, 0), (4, 2, 1025, 0)):
        assert det.lib.la_detector_features(det.handle, p(img), n, c, res, mod, p(out), s) != 0, (n, c, res, mod)
        assert det.lib.la_last_error()
    assert det.lib.la_detector_features(det.handle, p(img), 4, 2, 64, 1, p(out), s) == 0
    torch.cuda.synchronize()
    with pytest.raises(_lib.LatentAugmentError):
        det.features(img, modality=2)


def test_detector_leaves_engine_paths_unchanged(state):
    """A detector in the same process as an engine with the perceptual term and the projection targets: their losses and
    gradients stay at the run-to-run level of runs without it (those paths sum with atomics)."""
    from latentaugment_b200.engine import FeatureDetector, SynthesisEngine
    from oracle import lpips as olp
    from oracle import sg2
    res, C, batch = 64, 1, 4
    G = sg2.make_generator(seed=0, noise_strength=0.1, img_resolution=res, img_channels=C, channel_base=8192, channel_max=64)
    eng = SynthesisEngine(dict(G.state_dict()), img_resolution=res, img_channels=C, batch=batch, precision='bf16')
    eng.set_lpips(olp.random_vgg_state(7, olp.TAPS_SCRIPT), taps=olp.TAPS_SCRIPT, crop_size=64, per_sample_targets=True)
    img = _images(batch, C, res, 11).clamp(-1, 1)
    eng.set_projection_targets(_images(batch, C, res, 12).clamp(-1, 1))

    def run():
        pl, pg = eng.projection_loss_grad(img)
        eng.set_feature_bank(_images(6, C, 64, 13).clamp(-1, 1))
        ll, lg = eng.lpips_loss_grad(img, (0, 0), 1.0, norm_mode=0, centre=False)
        torch.cuda.synchronize()
        return [pl.clone(), pg.clone(), ll.reshape(1).clone(), lg.clone()]
    a, b = run(), run()
    base = [rel(x, y) for x, y in zip(a, b)]
    det = FeatureDetector(state, batch=8)
    det.features(_images(8, 1, 256, 14))
    c = run()
    after = [rel(x, y) for x, y in zip(c, a)]
    assert all(v <= 4 * w + 1e-6 for v, w in zip(after, base)), (after, base)


def test_precision_recall_from_images():
    """End to end from images: equal to the exhaustive definition on the GPU's own features; against the oracle's features
    every differing decision lies in the rounding band of the measured feature error."""
    from latentaugment_b200.engine import FeatureDetector
    from latentaugment_b200.metrics import precision_recall_images
    state = od.random_detector_state(7)
    det = FeatureDetector(state, batch=64, precision='fp32_parity')
    base = _images(1, 1, 64, 30)
    g = torch.Generator().manual_seed(31)
    real = (base + 0.5 * _images(200, 1, 64, 32)).clamp(-1, 1)
    gen = (base + 0.5 * _images(150, 1, 64, 33) + 0.1 * torch.randn([150, 1, 64, 64], generator=g)).clamp(-1, 1)
    stats = {}
    p, r = precision_recall_images(det, real, gen, 3, stats=stats)
    fr, fg = det.features(real).cpu(), det.features(gen).cpu()
    assert (p, r) == opr.definition_pr(fr, fg, 3)
    assert stats == {'fallback_precision': 0, 'fallback_recall': 0}
    orr, org = _oracle(state, real, 0).cpu(), _oracle(state, gen, 0).cpu()
    # tau: the largest relative change of any distance between the GPU's and the oracle's (fp16-rounded) features, plus one
    # fp16 rounding of the compared distances
    D = lambda a, b: opr.definition_sqdist(opr.as_definition_input(a), opr.as_definition_input(b)).double().clamp_min(0).sqrt()  # noqa: E731
    tau = 0.0
    for x, y, ox, oy in ((fg, fr, org, orr), (fr, fg, orr, org), (fr, fr, orr, orr), (fg, fg, org, org)):
        d, od_ = D(x, y), D(ox, oy)
        mask = od_ > 0
        tau = max(tau, float(((d - od_).abs()[mask] / od_[mask]).max()))
    tau += 2.0 ** -10
    decided = 0
    for name, man, probes, oman, oprobes in (('precision', fr, fg, orr, org), ('recall', fg, fr, org, orr)):
        mine = opr.definition_member(opr.as_definition_input(probes), opr.as_definition_input(man), opr.definition_radii(opr.as_definition_input(man), 3))
        ref = opr.definition_member(opr.as_definition_input(oprobes), opr.as_definition_input(oman),
                                    opr.definition_radii(opr.as_definition_input(oman), 3))
        band = opr.rounding_band(oprobes, oman, 3, tau)
        assert not ((mine != ref) & ~band).any(), (name, tau)
        decided += int((~band).sum())
    assert 0.0 < p < 1.0 or 0.0 < r < 1.0, (p, r)
    assert decided > 0, tau
