"""fp32 restatement of the VGG16 detector of precision / recall (DESIGN.md §13).

StyleGAN3's ``pr50k3`` embeds images with the NVIDIA VGG16 TorchScript (``return_features=True``: the 4096-d fc7 embedding).
That model cannot be read here, so the pin is torchvision's ``vgg16``: ``features`` -> ``avgpool`` (the identity at 7^2) ->
NCHW flatten -> ``classifier[:5]`` (fc6, ReLU, Dropout, fc7, ReLU; dropout is the identity in eval mode).

Per image, channel ``modality`` is quantised as StyleGAN3 saves generator output (``(x * 127.5 + 128).clamp(0, 255)`` to
uint8), replicated to three channels, area-resized to 224^2 and normalised with ``mean`` / ``std`` given in the 0..255 domain.
"""
import torch
import torch.nn.functional as F

from .lpips import CONV_IDX, VGG_CFG, random_vgg_state

IMAGENET_MEAN = tuple(255.0 * v for v in (0.485, 0.456, 0.406))
IMAGENET_STD = tuple(255.0 * v for v in (0.229, 0.224, 0.225))
SIZE = 224


def random_detector_state(seed=7):
    """``random_vgg_state(seed)``'s ``features.*`` entries plus He-scaled ``classifier.{0,3}.{weight,bias}`` from a separate
    generator (seeded ``seed + 1000``), so the convolution weights equal those of the perceptual-term tests."""
    sd = {k: v for k, v in random_vgg_state(seed).items() if k.startswith('features.')}
    g = torch.Generator().manual_seed(seed + 1000)
    for name, fan_in in (('classifier.0', 25088), ('classifier.3', 4096)):
        sd[f'{name}.weight'] = torch.randn([4096, fan_in], generator=g) * (2.0 / fan_in) ** 0.5
        sd[f'{name}.bias'] = torch.randn([4096], generator=g) * 0.05
    return sd


def quantise(x):
    """StyleGAN3's saved-image rule: [-1, 1] -> integer 0..255 (as fp32)."""
    return (x * 127.5 + 128).clamp(0, 255).to(torch.uint8).float()


def area_window_resize(u, size=SIZE):
    """The native input kernel's area rule restated for quantised (integer-valued) input: output (i, j) is the sum over rows
    [floor(i H / size), ceil((i + 1) H / size)) and the same columns, divided in fp32 by the window height, then its width.
    The kernel sums in fp32; a window of integers 0..255 sums exactly, so here the sums come from (exact) fp64 prefix sums."""
    n, c, H, W = u.shape
    assert torch.equal(u, u.round())
    idx = torch.arange(size)
    y0, y1 = idx * H // size, -(-(idx + 1) * H // size)
    x0, x1 = idx * W // size, -(-(idx + 1) * W // size)
    p = F.pad(u.double().cumsum(2).cumsum(3), (1, 0, 1, 0))
    s = (p[:, :, y1][:, :, :, x1] - p[:, :, y0][:, :, :, x1] - p[:, :, y1][:, :, :, x0] + p[:, :, y0][:, :, :, x0]).float()
    return s / (y1 - y0).float().view(1, 1, -1, 1) / (x1 - x0).float().view(1, 1, 1, -1)


def fc6_nhwc_weight(w6):
    """fc6 weights [4096, 25088] permuted from torchvision's NCHW flatten (c * 49 + h * 7 + w) to the NHWC order
    ((h * 7 + w) * 512 + c) of the pool5 tensor the native fc6 reads."""
    return w6.reshape(-1, 512, 49).permute(0, 2, 1).reshape(w6.shape[0], 25088)


def detector_input(img, modality=0, mean=IMAGENET_MEAN, std=IMAGENET_STD):
    """[n, C, H, W] in [-1, 1] -> the normalised [n, 3, 224, 224] network input."""
    u = quantise(img[:, modality:modality + 1].float())
    v = F.interpolate(u, size=(SIZE, SIZE), mode='area')
    m = torch.tensor(mean, dtype=v.dtype, device=v.device).view(1, 3, 1, 1)
    s = torch.tensor(std, dtype=v.dtype, device=v.device).view(1, 3, 1, 1)
    return (v.expand(-1, 3, -1, -1) - m) / s


def network(state, x):
    """torchvision vgg16 ``features`` + flatten + ``classifier[:5]`` (eval) on a normalised [n, 3, 224, 224] input."""
    ci = 0
    for v in VGG_CFG + ['M']:
        if v == 'M':
            x = F.max_pool2d(x, 2, 2)
            continue
        i = CONV_IDX[ci]
        x = F.relu(F.conv2d(x, state[f'features.{i}.weight'], state[f'features.{i}.bias'], padding=1))
        ci += 1
    x = F.adaptive_avg_pool2d(x, (7, 7)).flatten(1)
    x = F.relu(F.linear(x, state['classifier.0.weight'], state['classifier.0.bias']))
    return F.relu(F.linear(x, state['classifier.3.weight'], state['classifier.3.bias']))


def detector_features(state, img, modality=0, mean=IMAGENET_MEAN, std=IMAGENET_STD):
    """fp32 [n, 4096] fc7 embeddings of channel ``modality`` of ``img`` (computed on ``img``'s device)."""
    state = {k: v.to(img.device, torch.float32) for k, v in state.items()}
    return network(state, detector_input(img, modality, mean, std))
