"""Host side of the projection of real images into W (StyleGAN2-ADA ``projector.py::project``, batched; DESIGN.md
"Projection"): the per-step learning-rate and w-noise schedule and the ``w_avg`` / ``w_std`` statistics.  The schedule is
one function so the engine wrapper and the oracle cannot drift apart."""
import math

import numpy as np

# upstream projector.py defaults
NUM_STEPS = 1000
INITIAL_LR = 0.1
INITIAL_NOISE_FACTOR = 0.05
LR_RAMPDOWN_LENGTH = 0.25
LR_RAMPUP_LENGTH = 0.05
NOISE_RAMP_LENGTH = 0.75
W_AVG_SAMPLES = 10000
W_AVG_SEED = 123


def projection_schedule(num_steps=NUM_STEPS, *, initial_lr=INITIAL_LR, initial_noise_factor=INITIAL_NOISE_FACTOR,
                        lr_rampdown_length=LR_RAMPDOWN_LENGTH, lr_rampup_length=LR_RAMPUP_LENGTH,
                        noise_ramp_length=NOISE_RAMP_LENGTH):
    """(lr [T], sigma_unit [T]) as float64 arrays.  With tau = t / T:
    ``sigma_unit = initial_noise_factor * max(0, 1 - tau / noise_ramp_length)^2`` (multiply by ``w_std`` for the w noise),
    ``lr = initial_lr * (0.5 - 0.5 cos(pi * min(1, (1 - tau) / lr_rampdown_length))) * min(1, tau / lr_rampup_length)``,
    so ``lr[0] = 0`` as upstream."""
    T = int(num_steps)
    lr = np.zeros(T, dtype=np.float64)
    sigma = np.zeros(T, dtype=np.float64)
    for t in range(T):
        tau = t / T
        sigma[t] = initial_noise_factor * max(0.0, 1.0 - tau / noise_ramp_length) ** 2
        ramp = min(1.0, (1.0 - tau) / lr_rampdown_length)
        ramp = 0.5 - 0.5 * math.cos(ramp * math.pi)
        ramp = ramp * min(1.0, tau / lr_rampup_length)
        lr[t] = initial_lr * ramp
    return lr, sigma


def w_avg_z(z_dim, n=W_AVG_SAMPLES, seed=W_AVG_SEED):
    """The ``z`` samples behind ``w_avg`` / ``w_std``: ``np.random.RandomState(123).randn(10000, z_dim)`` (projector.py)."""
    return np.random.RandomState(seed).randn(n, z_dim)


def w_stats_from_samples(w):
    """``w`` [n, w_dim] (row 0 of the mapped samples) -> (w_avg [w_dim], w_std scalar) in float64:
    ``w_std = sqrt(sum ||w - w_avg||^2 / n)``."""
    w = np.asarray(w, dtype=np.float64)
    avg = w.mean(0)
    std = float(np.sqrt(((w - avg) ** 2).sum() / w.shape[0]))
    return avg, std


def area_downsample_factor(img_resolution):
    """The projection window is the whole image; above 256 it is area-downsampled 2x (upstream's ``> 256`` rule).
    Resolutions above 512 are refused."""
    if img_resolution > 512:
        raise ValueError(f'projection supports resolutions up to 512 (got {img_resolution})')
    return 2 if img_resolution > 256 else 1
