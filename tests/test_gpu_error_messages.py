"""A rejected discriminator or perceptual-term descriptor fails la_set_discriminator / la_set_lpips with -6 / -7, and the
la_last_error() text names the module that rejected it exactly once."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu


def test_rejected_descriptors_name_their_module_once():
    from latentaugment_b200 import _lib
    from latentaugment_b200.engine import SynthesisEngine
    from oracle import synthetic
    wl = synthetic.make_workload('tiny')
    G = wl['G']
    eng = SynthesisEngine(dict(G.state_dict()), img_resolution=G.img_resolution, img_channels=G.img_channels, w_dim=G.w_dim,
                          z_dim=G.z_dim, batch=wl['w0'].shape[0], precision='bf16')
    ws = torch.empty(1 << 20, dtype=torch.uint8, device='cuda')
    base = C.c_void_p((ws.data_ptr() + 1023) // 1024 * 1024)
    nbytes = (1 << 20) - 1024
    torch.cuda.synchronize()

    d = _lib.DiscDesc()
    d.img_resolution, d.img_channels = G.img_resolution, G.img_channels
    d.num_blocks = G.img_resolution.bit_length() - 3                  # 8 << (num_blocks - 1) == resolution
    for b in range(d.num_blocks + 1):
        d.channels[b] = 64
    d.conv_clamp, d.mbstd_group_size = 256.0, 9                        # the group must be 1..8
    assert eng.lib.la_set_discriminator(eng.handle, C.byref(d), base, nbytes, None) == -6
    msg = eng.lib.la_last_error().decode()
    assert 'mbstd_group_size' in msg and msg.count('discriminator') == 1, msg

    v = _lib.VggDesc()
    v.crop_size = 48                                                   # a power of two >= 64
    for k in range(3):
        v.std[k] = 1.0
    assert eng.lib.la_set_lpips(eng.handle, C.byref(v), base, nbytes, None) == -7
    msg = eng.lib.la_last_error().decode()
    assert 'crop_size' in msg and msg.count('lpips') == 1, msg
