"""Benchmark of the VGG16 detector (DESIGN.md §13): fc7 embeddings of one set of 50 000 images, native detector in both
precisions against torchvision's vgg16 on the same GPU and the same images.

    python tools/bench_detector.py [--n 50000] [--res 256] [--out profiles/detector_bench_n1.json]

The images are seeded 256^2 one-modality images generated chunk by chunk on the device (outside the timed windows); each
configuration is warmed up on one chunk, then timed over the whole set with CUDA events around each chunk's embedding.
The comparator is torchvision's vgg16 (features, avgpool, classifier[:5]) with the same weights and the same input
pipeline (quantise, area interpolate to 224^2, normalise), in fp32 with TF32 off and with TF32 on.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

from oracle import detector as od

CHUNK = 256


def flops_per_image(cin_first):
    """(conv, fc) FLOPs per image at 224^2, 2 per multiply-add; the first convolution with `cin_first` input channels."""
    cout = [64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512, 512]
    cin = [cin_first] + cout[:-1]
    res = [224, 224, 112, 112, 56, 56, 56, 28, 28, 28, 14, 14, 14]
    conv = sum(2 * 9 * ci * co * r * r for ci, co, r in zip(cin, cout, res))
    fc = 2 * (25088 * 4096 + 4096 * 4096)
    return conv, fc


def chunk_images(i, n, res, dev):
    g = torch.Generator(device=dev).manual_seed(1000 + i)
    low = torch.randn([n, 1, 8, 8], generator=g, device=dev)
    low = torch.nn.functional.interpolate(low, size=(res, res), mode='bilinear', align_corners=False)
    return (0.6 * low + 0.3 * torch.randn([n, 1, res, res], generator=g, device=dev)).clamp(-1, 1)


def time_set(embed, n, res, dev):
    embed(chunk_images(0, CHUNK, res, dev))                # warm-up
    torch.cuda.synchronize(dev)
    total = 0.0
    for i, b in enumerate(range(0, n, CHUNK)):
        x = chunk_images(i, min(CHUNK, n - b), res, dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        embed(x)
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1) / 1e3
    return total


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        name, power = [s.strip() for s in q.stdout.strip().splitlines()[0].split(',')]
        return name, power
    except Exception as e:      # the torch name stands in; the power limit is then unknown
        return torch.cuda.get_device_name(), f'unavailable ({e})'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=50000)
    ap.add_argument('--res', type=int, default=256)
    ap.add_argument('--out', default='profiles/detector_bench_n1.json')
    a = ap.parse_args()
    import torchvision

    from latentaugment_b200.engine import FeatureDetector
    dev = torch.device('cuda:0')
    name, power = gpu_info()
    state = od.random_detector_state(7)
    conv3, fc = flops_per_image(3)
    conv64, _ = flops_per_image(64)
    res = {'gpu': name, 'power_limit': power, 'n_images': a.n, 'res': a.res, 'chunk': CHUNK,
           'gflop_per_image': {'conv_cin3': conv3 / 1e9, 'fc': fc / 1e9, 'conv_executed_cin64': conv64 / 1e9}}
    probe = chunk_images(0, CHUNK, a.res, dev)

    vgg = torchvision.models.vgg16(weights=None)
    vgg.load_state_dict({**vgg.state_dict(), **state})
    vgg = vgg.to(dev).eval()

    def torch_embed(x):
        with torch.no_grad():
            f = vgg.features(od.detector_input(x))
            return vgg.classifier[:5](torch.flatten(vgg.avgpool(f), 1))
    refs = {}
    for tf32 in (False, True):
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = tf32
        key = 'torchvision_fp32_tf32' if tf32 else 'torchvision_fp32'
        t = time_set(torch_embed, a.n, a.res, dev)
        refs[key] = torch_embed(probe)
        res[key] = {'seconds_per_set': t, 'tflops_algorithmic': a.n * (conv3 + fc) / t / 1e12}
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    for prec in ('bf16', 'fp32_parity'):
        det = FeatureDetector(state, batch=CHUNK, precision=prec, device=dev)
        t = time_set(det.features, a.n, a.res, dev)
        f = det.features(probe)
        res[prec] = {'seconds_per_set': t, 'tflops_algorithmic': a.n * (conv3 + fc) / t / 1e12,
                     'tflops_executed': a.n * (conv64 + fc) / t / 1e12,
                     'rel_l2_vs_torchvision_fp32': float((f - refs['torchvision_fp32']).double().norm() / refs['torchvision_fp32'].double().norm()),
                     'rel_l2_vs_torchvision_tf32': float((f - refs['torchvision_fp32_tf32']).double().norm() / refs['torchvision_fp32_tf32'].double().norm())}
        del det
    res['speedup_bf16_vs_tf32'] = res['torchvision_fp32_tf32']['seconds_per_set'] / res['bf16']['seconds_per_set']
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=2)


if __name__ == '__main__':
    main()
