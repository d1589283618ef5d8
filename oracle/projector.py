"""Oracle restatement of the projection of real images into W.  TEST INFRASTRUCTURE (see oracle/__init__.py).

The algorithm is StyleGAN2-ADA ``projector.py::project``, batched, with the three differences DESIGN.md "Projection"
defines: the noise maps stay at ``noise_const`` and are not optimised (no noise regulariser); the VGG input follows the
perceptual term (each modality replicated to 3 channels, z-scored, all five taps with their lin weights); images above
256 are area-downsampled 2x.  The schedule is ``latentaugment_b200.projection.projection_schedule``, the same function
the engine wrapper calls.

Runs in the dtype of ``targets`` (float64 for the algebraic checks: the generator is copied to that dtype).
"""
import copy

import torch
import torch.nn.functional as F

from latentaugment_b200.projection import projection_schedule, w_avg_z, w_stats_from_samples
from . import lpips as olp
from . import ops


def synthesize(G, ws):
    """``G.synthesis(ws, noise_mode='const')`` without the float32 casts of ``Synthesis.forward`` (dtype follows G / ws)."""
    S = G.synthesis
    x = img = None
    idx = 0
    for r in S.block_resolutions:
        blk = getattr(S, f'b{r}')
        wi = iter(ws.narrow(1, idx, blk.num_conv + blk.num_torgb).unbind(dim=1))
        x = blk.const.unsqueeze(0).repeat([ws.shape[0], 1, 1, 1]) if blk.cin == 0 else blk.conv0(x, next(wi), noise_mode='const')
        x = blk.conv1(x, next(wi), noise_mode='const')
        if img is not None:
            img = ops.upsample2d(img, blk.resample_filter)
        y = blk.torgb(x, next(wi))
        img = y if img is None else img + y
        idx += blk.num_conv
    return img


def w_stats(G):
    """(w_avg [w_dim], w_std) from ``RandomState(123)`` z through the mapping at psi = 1, row 0 (float64 numpy)."""
    with torch.no_grad():
        z = torch.from_numpy(w_avg_z(G.z_dim)).float()
        w = G.mapping(z, None)[:, 0]
    return w_stats_from_samples(w.double().numpy())


def per_sample_distance(vgg_state, x, y_feats, taps=olp.TAPS_SCRIPT):
    """x [B, C, R, R] -> [B]: sum over modalities and taps of (1/P) sum_p sum_c w_c (n^_x - n^_y)^2, y_feats[c] = target taps."""
    if x.shape[-1] > 256:
        x = F.avg_pool2d(x, 2)
    lw = olp.lin_weights(vgg_state, taps)
    d = 0.0
    for c in range(x.shape[1]):
        fx = olp.vgg_features(vgg_state, x[:, c:c + 1].repeat(1, 3, 1, 1), taps)
        for a, b, w in zip(fx, y_feats[c], lw):
            d = d + ((a - b) ** 2 * w.to(a).reshape(1, -1, 1, 1)).sum(1).mean((1, 2))
    return d


def target_features(vgg_state, y, taps=olp.TAPS_SCRIPT):
    if y.shape[-1] > 256:
        y = F.avg_pool2d(y, 2)
    with torch.no_grad():
        return [olp.vgg_features(vgg_state, y[:, c:c + 1].repeat(1, 3, 1, 1), taps) for c in range(y.shape[1])]


def project(G, vgg_state, targets, w_noise, *, w_avg, w_std, num_steps, taps=olp.TAPS_SCRIPT, w0=None, **schedule):
    """targets [B, C, R, R] in [-1, 1]; w_noise [T, B, w_dim] unit normal.  Returns (w [B, w_dim], per-step loss [T] float64).
    cuDNN runs in its deterministic mode here, so the same inputs give the same trajectory in every run."""
    saved = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        return _project(G, vgg_state, targets, w_noise, w_avg, w_std, num_steps, taps, w0, schedule)
    finally:
        torch.backends.cudnn.deterministic = saved


def _project(G, vgg_state, targets, w_noise, w_avg, w_std, num_steps, taps, w0, schedule):
    dt = targets.dtype
    G = copy.deepcopy(G).to(dt)
    st = {k: v.to(dt) for k, v in vgg_state.items()}
    y_feats = target_features(st, targets, taps)
    B = targets.shape[0]
    lr, sigma = projection_schedule(num_steps, **schedule)
    w0 = torch.as_tensor(w_avg, dtype=dt).reshape(1, -1).repeat(B, 1) if w0 is None else w0.to(dt).clone()
    w_opt = w0.to(targets.device).requires_grad_(True)
    opt = torch.optim.Adam([w_opt], betas=(0.9, 0.999), lr=0.1, eps=1e-8)
    losses = []
    for t in range(num_steps):
        for grp in opt.param_groups:
            grp['lr'] = float(lr[t])
        ws = (w_opt + float(w_std * sigma[t]) * w_noise[t].to(dt)).unsqueeze(1).repeat(1, G.num_ws, 1)
        loss = per_sample_distance(st, synthesize(G, ws), y_feats, taps).sum()
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    return w_opt.detach(), torch.tensor(losses, dtype=torch.float64)
