"""Seeded synthetic workloads (SURVEY.md §8d) shared by the golden generator, the
parity tests and the CPU-baseline leg of bench.py.  TEST INFRASTRUCTURE.

Everything is drawn on the CPU with explicit ``torch.Generator`` seeds so the same
tensors can be rebuilt on the GPU box without shipping them.
"""
import torch

from . import sg2

# name -> generator kwargs + workload sizes.  "c1"/"c2"/"c3" are BASELINE.json's
# configs[0..2]; "tiny*" are reduced cases the CPU oracle finishes in seconds.
CONFIGS = {
    'tiny': dict(img_resolution=32, img_channels=2, channel_base=2048, channel_max=64,
                 batch=4, steps=3, bank=64, img_bank=8),
    'tiny128': dict(img_resolution=16, img_channels=3, channel_base=2048, channel_max=128,
                    batch=8, steps=2, bank=32, img_bank=4),
    'small': dict(img_resolution=64, img_channels=3, channel_base=8192, channel_max=128,
                  batch=2, steps=2, bank=32, img_bank=4),
    'c1': dict(img_resolution=128, img_channels=1, channel_base=32768, channel_max=512,
               batch=4, steps=5, bank=256, img_bank=64),
    'c2': dict(img_resolution=256, img_channels=3, channel_base=32768, channel_max=512,
               batch=32, steps=10, bank=4096, img_bank=64),
    'c3': dict(img_resolution=512, img_channels=3, channel_base=32768, channel_max=512,
               batch=128, steps=10, bank=4096, img_bank=64),
}


def generator_kwargs(cfg):
    c = CONFIGS[cfg] if isinstance(cfg, str) else cfg
    return dict(img_resolution=c['img_resolution'], img_channels=c['img_channels'],
                channel_base=c['channel_base'], channel_max=c['channel_max'])


def _randn(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


def make_workload(cfg, noise_strength=0.0, batch=None, with_img_bank=True, conv_clamp=256.0):
    """Returns dict(G, W [M,num_ws,w_dim], w0 [B,1,w_dim], X [Mi,C,res,res] or None).  ``conv_clamp`` changes no drawn
    tensor."""
    c = dict(CONFIGS[cfg]) if isinstance(cfg, str) else dict(cfg)
    B = batch if batch is not None else c['batch']
    G = sg2.make_generator(seed=0, noise_strength=noise_strength, conv_clamp=conv_clamp, **generator_kwargs(c))
    with torch.no_grad():
        W = G.mapping(_randn([c['bank'], G.z_dim], 1), None)[:, :1].repeat(1, G.num_ws, 1).contiguous()
        w0 = G.mapping(_randn([B, G.z_dim], 2), None)[:, :1].contiguous()
    X = None
    if with_img_bank:
        X = torch.rand([c['img_bank'], c['img_channels'], c['img_resolution'], c['img_resolution']],
                       generator=torch.Generator().manual_seed(3)) * 2 - 1
    return dict(G=G, W=W, w0=w0, X=X, cfg=c)
