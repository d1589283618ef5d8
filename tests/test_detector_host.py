"""Host-side checks of the VGG16 detector (DESIGN.md §13): the oracle against torchvision's vgg16, the quantise, area and fc6
permutation rules the native kernels implement, the C-ABI planner and rejections (no device needed), the sharded
``metrics.precision_recall_images`` under a 2-rank gloo group, and the tolerance basis the GPU test's tolerances rest on."""
import ctypes
import importlib.util
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN, rel_l2
from oracle import detector as od
from oracle import precision_recall as opr


@pytest.fixture(scope='module')
def state():
    return od.random_detector_state(7)


def _images(n, C, res, seed):
    g = torch.Generator().manual_seed(seed)
    low = F.interpolate(torch.randn([n, C, 8, 8], generator=g), size=(res, res), mode='bilinear', align_corners=False)
    return (0.6 * low + 0.3 * torch.randn([n, C, res, res], generator=g)).clamp(-1.1, 1.1)


def test_random_detector_state_extends_the_perceptual_state(state):
    from oracle.lpips import random_vgg_state
    vgg = random_vgg_state(7)
    assert all(torch.equal(state[k], v) for k, v in vgg.items() if k.startswith('features.'))
    assert sorted(k for k in state if not k.startswith('features.')) == sorted(f'classifier.{i}.{p}' for i in (0, 3) for p in ('weight', 'bias'))
    assert torch.equal(random_vgg_state(7)['lin.0.weight'], vgg['lin.0.weight'])        # its random stream is unchanged


@pytest.mark.parametrize('res', [64, 224, 256, 512])
def test_oracle_equals_torchvision_vgg16(state, res):
    import torchvision
    vgg = torchvision.models.vgg16(weights=None)
    vgg.load_state_dict({**vgg.state_dict(), **state})
    vgg.eval()
    img = _images(2, 2, res, res)
    with torch.no_grad():
        for c in range(2):
            x = od.detector_input(img, c)
            ref = vgg.classifier[:5](torch.flatten(vgg.avgpool(vgg.features(x)), 1))
            got = od.detector_features(state, img, c)
            assert rel_l2(got, ref) < 1e-6, (res, c)


def test_quantise_round_trips_the_golden_image_zip():
    from latentaugment_b200.augments.utils.util_dataset import ImgDataset
    ds = ImgDataset(os.path.join(GOLDEN, 'formats', 'images.zip'), 'train', ['MR_nonrigid_CT', 'MR_MR_T2'], resolution=8)
    u = np.stack([ds[i][0] for i in range(len(ds))])
    assert np.array_equal(u, np.round(u)) and u.min() >= 0 and u.max() <= 255 and len(np.unique(u)) > 20
    x = torch.from_numpy(u / 127.5 - 1)                     # what the zip loader hands to the loop (util_dataset.py)
    assert x.dtype == torch.float32
    assert torch.equal(od.quantise(x), torch.from_numpy(u))
    assert torch.equal(od.quantise(torch.tensor([-1.5, -1.0, 1.0, 1.5, 0.0])), torch.tensor([0.0, 0.0, 255.0, 255.0, 128.0]))


@pytest.mark.parametrize('res', [64, 128, 224, 256, 512])
def test_area_window_rule_is_interpolate_area_bit_for_bit(res):
    u = od.quantise(_images(2, 1, res, 40 + res))
    assert torch.equal(od.area_window_resize(u), F.interpolate(u, size=(224, 224), mode='area'))


def test_fc6_permutation_equals_linear_on_the_nchw_flatten():
    g = torch.Generator().manual_seed(3)
    w = torch.randint(-8, 9, [64, 25088], generator=g).float()        # small integers: every sum is exact in fp32
    x = torch.randint(0, 5, [3, 512, 7, 7], generator=g).float()
    nhwc = x.permute(0, 2, 3, 1).reshape(3, 25088)
    assert torch.equal(F.linear(nhwc, od.fc6_nhwc_weight(w)), F.linear(x.flatten(1), w))


def _desc(ptr=1024, skip=None):
    from latentaugment_b200 import _lib
    d = _lib.DetectorDesc()
    for i in range(13):
        d.d_conv_weight[i] = d.d_conv_bias[i] = ctypes.c_void_p(ptr)
    for f in ('d_fc6_weight', 'd_fc6_bias', 'd_fc7_weight', 'd_fc7_bias'):
        setattr(d, f, ctypes.c_void_p(0 if f == skip else ptr))
    for k in range(3):
        d.mean[k], d.std[k] = od.IMAGENET_MEAN[k], od.IMAGENET_STD[k]
    return d


def test_detector_planner_and_rejections_on_the_host():
    from latentaugment_b200 import _lib
    lib = _lib.load()
    n = ctypes.c_size_t(0)
    d = _desc()
    assert lib.la_detector_workspace_bytes(ctypes.byref(d), 256, 0, ctypes.byref(n)) == 0
    act = 2 * 256 * 224 * 224 * 64 * 2                                 # two ping-pong buffers, bf16
    weights = (4096 * 25088 + 4096 * 4096 + 15_000_000) * 2          # fc6 + fc7 + the padded convolutions (upper bound)
    assert act < n.value < act + weights + 16 * 2 ** 20
    bf16 = n.value
    assert lib.la_detector_workspace_bytes(ctypes.byref(d), 256, 1, ctypes.byref(n)) == 0
    assert 2 * bf16 - 16 * 2 ** 20 < n.value < 2 * bf16               # split: every bf16 operand has a lo plane
    for skip in ('d_fc6_weight', 'd_fc6_bias', 'd_fc7_weight', 'd_fc7_bias'):
        assert lib.la_detector_workspace_bytes(ctypes.byref(_desc(skip=skip)), 4, 0, ctypes.byref(n)) != 0, skip
        assert b'fc' in lib.la_last_error()
    assert lib.la_detector_workspace_bytes(ctypes.byref(d), 0, 0, ctypes.byref(n)) != 0          # batch
    assert lib.la_detector_workspace_bytes(ctypes.byref(d), 4, 2, ctypes.byref(n)) != 0          # precision
    bad = _desc()
    bad.std[1] = 0.0
    assert lib.la_detector_workspace_bytes(ctypes.byref(bad), 4, 0, ctypes.byref(n)) != 0
    # creation rejects a short or misaligned workspace and missing weights before touching the device
    assert lib.la_detector_workspace_bytes(ctypes.byref(d), 4, 0, ctypes.byref(n)) == 0
    base = 1 << 30
    h = ctypes.c_void_p()
    assert lib.la_detector_create(ctypes.byref(d), 4, 0, ctypes.c_void_p(base), n.value - 1, None, ctypes.byref(h)) != 0
    assert b'too small' in lib.la_last_error()
    assert lib.la_detector_create(ctypes.byref(d), 4, 0, ctypes.c_void_p(base + 8), 2 * n.value, None, ctypes.byref(h)) != 0
    assert b'aligned' in lib.la_last_error()
    assert lib.la_detector_create(ctypes.byref(_desc(skip='d_fc7_weight')), 4, 0, ctypes.c_void_p(base), 2 * n.value, None,
                                  ctypes.byref(h)) != 0
    assert not h.value
    assert lib.la_detector_features(None, ctypes.c_void_p(base), 1, 1, 64, 0, ctypes.c_void_p(base), None) != 0


class _StandInDetector:
    """FeatureDetector stand-in on the CPU: a fixed random projection of the quantised, area-resized modality, recording
    how many images each call embeds."""
    calls = []

    def __init__(self):
        self.w = torch.randn([64 * 64, 128], generator=torch.Generator().manual_seed(8)) / 64

    def features(self, img, modality=0):
        _StandInDetector.calls.append(img.shape[0])
        u = F.interpolate(od.quantise(img[:, modality:modality + 1]), size=(64, 64), mode='area')
        return torch.relu(u.flatten(1) / 255 @ self.w)


def _pri_worker(rank, world, port, q):
    import torch.distributed as dist

    from latentaugment_b200 import metrics, parallel
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    gathers = []
    ag = dist.all_gather_into_tensor
    dist.all_gather_into_tensor = lambda *a, **k: (gathers.append(1), ag(*a, **k))[1]
    real, gen = _images(53, 2, 96, 1).clamp(-1, 1), _images(41, 2, 96, 2).clamp(-1, 1)
    det = _StandInDetector()
    seen = {}

    def precision_recall(r, g, nhood_size, group=None, stats=None):       # the metric itself: its inputs are what is checked
        seen['shapes'] = (tuple(r.shape), tuple(g.shape))
        return opr.definition_pr(r, g, nhood_size)
    metrics.precision_recall = precision_recall
    p, r = metrics.precision_recall_images(det, real, gen, 3, modality=1)
    ref = _StandInDetector()
    p0, r0 = opr.definition_pr(ref.features(real, 1), ref.features(gen, 1), 3)
    expect = [parallel.shard_range(53, rank, world)[1] - parallel.shard_range(53, rank, world)[0],
              parallel.shard_range(41, rank, world)[1] - parallel.shard_range(41, rank, world)[0]]
    ok = (p, r) == (p0, r0) and _StandInDetector.calls[:2] == expect and len(gathers) == 2 and seen['shapes'] == ((53, 128), (41, 128))
    q.put((rank, bool(ok), (p, r, p0, r0, _StandInDetector.calls, len(gathers), seen)))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_precision_recall_images_gloo_world2():
    """Each rank embeds its shard_range of each image set; one all_gather_into_tensor per set gives every rank the whole
    features, so the metric sees exactly the single-process features."""
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 35500 + os.getpid() % 2000
    procs = [ctx.Process(target=_pri_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert [(r, ok) for r, ok, _ in res] == [(0, True), (1, True)], res


def test_tolerance_basis(state):
    """Perturbing every weight by a relative 2^-9 (bf16) and 2^-17 (split operands) moves the features by the relative L2
    recorded as BASIS_BF16 / BASIS_SPLIT in tests/test_gpu_detector.py (within 30 %)."""
    spec = importlib.util.spec_from_file_location('gpu_det', os.path.join(os.path.dirname(__file__), 'test_gpu_detector.py'))
    gpu = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gpu)
    img = _images(3, 1, 64, 3)
    f0 = od.detector_features(state, img)
    for eps, recorded in ((2.0 ** -9, gpu.BASIS_BF16), (2.0 ** -17, gpu.BASIS_SPLIT)):
        vals = []
        for draw in range(2):
            g = torch.Generator().manual_seed(100 + draw)
            sp = {k: v * (1 + eps * (torch.randint(0, 2, v.shape, generator=g) * 2 - 1)) for k, v in state.items()}
            vals.append(rel_l2(od.detector_features(sp, img), f0))
        assert 0.7 * recorded < max(vals) < 1.3 * recorded, (eps, vals, recorded)
