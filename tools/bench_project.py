"""Projection throughput at the C2 shape (256 x 256, 3 modalities, batch 32; DESIGN.md "Projection"): one JSON line with,
per precision, ms per projection step, projected images/s at T = 1000 steps, the algorithmic FLOPs of one step and the
achieved rate, plus the device name and power limit read in the same run.

    python tools/bench_project.py [--steps 20] [--warmup 3] [--precision fp32_parity,bf16]

ms per step = (time of a `steps`-step projection - time of a `steps/2`-step one) / (steps - steps/2): the per-call setup
(schedule, its copies to the device, the first perturbed code) is not projection work and cancels.

FLOPs per step are computed from shapes: generator forward + data gradient = 2 * F_syn * B (F_syn: the forward
multiply-adds x 2 of one sample: 3x3 modulated convs, up-sampling convs as stride-2 transposed convs (9 taps per input
pixel), toRGB),
VGG16 forward + data gradient = 2 * F_vgg * B * C over the B * C whole-image windows.  Seeded random weights.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

import torch  # noqa: E402

VGG = [(3, 64), (64, 64), 'M', (64, 128), (128, 128), 'M', (128, 256), (256, 256), (256, 256), 'M', (256, 512), (512, 512), (512, 512), 'M',
       (512, 512), (512, 512), (512, 512)]


def synthesis_flops(res, C, channel_base=32768, channel_max=512):
    """Forward FLOPs (2 x multiply-adds) of one sample's synthesis."""
    f, r, prev = 0, 4, None
    while r <= res:
        ch = min(channel_base // r, channel_max)
        if prev is not None:
            f += 2 * (r // 2) ** 2 * 9 * prev * ch  # conv0: x2 up as a stride-2 transposed conv (9 taps per input pixel)
        f += 2 * r * r * 9 * ch * ch              # conv1
        f += 2 * r * r * ch * C                   # toRGB
        prev, r = ch, r * 2
    return f


def vgg_flops(win):
    f, r = 0, win
    for layer in VGG:
        if layer == 'M':
            r //= 2
        else:
            f += 2 * r * r * 9 * layer[0] * layer[1]
    return f


def power_limit():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader,nounits', '-i', str(torch.cuda.current_device())],
                             capture_output=True, text=True, timeout=30)
        return float(out.stdout.strip().splitlines()[0])
    except Exception:       # noqa: BLE001 -- reported as unknown
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--precision', default='fp32_parity,bf16')
    ap.add_argument('--batch', type=int, default=32)
    ap.add_argument('--res', type=int, default=256)
    ap.add_argument('--channels', type=int, default=3)
    args = ap.parse_args()
    from latentaugment_b200.engine import SynthesisEngine
    from latentaugment_b200.utils import synthetic
    res, C, B = args.res, args.channels, args.batch
    win = min(res, 256)
    f_step = 2 * synthesis_flops(res, C) * B + 2 * vgg_flops(win) * B * C
    G = synthetic.random_generator_state(img_resolution=res, img_channels=C)
    vgg = synthetic.random_vgg_state(7, (4, 9, 16, 23, 30))
    y = torch.rand([B, C, res, res], generator=torch.Generator().manual_seed(3)) * 2 - 1
    out = dict(metric='projection', shape=dict(res=res, img_channels=C, batch=B, window=win), steps=args.steps,
               device=torch.cuda.get_device_name(), power_limit_w=power_limit(),
               flops_per_step=f_step, flops_generator=2 * synthesis_flops(res, C) * B, flops_vgg=2 * vgg_flops(win) * B * C)
    for prec in args.precision.split(','):
        eng = SynthesisEngine(G, img_resolution=res, img_channels=C, batch=B, precision=prec)
        eng.set_lpips(vgg, taps=(4, 9, 16, 23, 30), crop_size=win, per_sample_targets=True)
        eng.set_projection_targets(y)
        noise = torch.randn([args.steps, B, eng.w_dim], generator=torch.Generator().manual_seed(0)).cuda()
        eng.project(num_steps=args.warmup, w_noise=noise[:args.warmup])          # w_stats, graph capture

        def timed(k):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.project(num_steps=k, w_noise=noise[:k])
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b)
        # a call's fixed part (schedule, its host-to-device copies, setup kernels) cancels in the difference of two lengths
        half = args.steps // 2
        ms = (timed(args.steps) - timed(half)) / (args.steps - half)
        eng.debug_check()
        out[prec] = dict(ms_per_step=round(ms, 3), images_per_s_at_1000_steps=round(B / (ms * 1e-3 * 1000), 3),
                         tflops=round(f_step / (ms * 1e-3) / 1e12, 1))
        del eng
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == '__main__':
    main()
