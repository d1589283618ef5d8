"""CPU checks of the projection into W (DESIGN.md "Projection"): the oracle's algebra, the shared schedule, the tolerance
basis of tests/test_gpu_projection.py, the inverted-code zip writer with a stand-in engine, and the workspace plan of the
per-sample target features."""
import ctypes as C
import math
import os
import pickle
import zipfile

import numpy as np
import pytest
import torch

TAPS = (4, 9, 16, 23, 30)


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def _small(res=64, C=3, cb=8192, cm=128):
    from oracle import sg2
    return sg2.make_generator(seed=0, noise_strength=0.1, img_resolution=res, img_channels=C, channel_base=cb, channel_max=cm)


def _targets(G, B, seed, dtype=torch.float32):
    with torch.no_grad():
        w = G.mapping(torch.randn([B, G.z_dim], generator=torch.Generator().manual_seed(seed)), None)
        return G.synthesis(w, noise_mode='const').clamp(-1, 1).to(dtype)


def test_batched_projection_equals_single_projections_in_fp64():
    from oracle import lpips as olp
    from oracle import projector as opj
    G = _small(C=1, cb=4096, cm=64)
    st = olp.random_vgg_state(7, TAPS)
    wa, ws = opj.w_stats(G)
    B, T = 3, 6
    y = _targets(G, B, 9, torch.float64)
    n = torch.randn([T, B, G.w_dim], generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    w, loss = opj.project(G, st, y, n, w_avg=wa, w_std=ws, num_steps=T)
    singles = [opj.project(G, st, y[i:i + 1], n[:, i:i + 1], w_avg=wa, w_std=ws, num_steps=T) for i in range(B)]
    w1 = torch.cat([s[0] for s in singles])
    l1 = sum(s[1] for s in singles)
    print(f'\nbatched vs single: w max-rel {float((w - w1).abs().max() / w1.abs().max()):.2e}, loss rel {_rel(loss, l1):.2e}')
    assert float((w - w1).abs().max() / w1.abs().max()) <= 1e-12
    assert _rel(loss, l1) <= 1e-12
    assert float((w - torch.as_tensor(wa)).abs().max()) > 1e-3        # the codes moved


def test_projection_schedule_closed_form_and_shared():
    import latentaugment_b200.engine as eng_mod
    from latentaugment_b200 import projection
    from oracle import projector as opj
    assert opj.projection_schedule is projection.projection_schedule is eng_mod._proj.projection_schedule
    T = 1000
    lr, sig = projection.projection_schedule(T)
    assert lr.shape == sig.shape == (T,)
    assert lr[0] == 0.0 and sig[0] == 0.05
    # tau = 0.05: ramp-up complete, ramp-down not started
    assert lr[50] == pytest.approx(0.1, abs=1e-15)
    assert sig[50] == pytest.approx(0.05 * (1 - 0.05 / 0.75) ** 2, rel=1e-15)
    # tau = 0.75: noise has ramped to 0; lr still 0.1 (ramp-down starts at 1 - 0.25)
    assert sig[750] == 0.0 and lr[750] == pytest.approx(0.1, abs=1e-15)
    tau = (T - 1) / T
    assert lr[T - 1] == pytest.approx(0.1 * (0.5 - 0.5 * math.cos(math.pi * (1 - tau) / 0.25)), rel=1e-13)
    assert sig[T - 1] == 0.0
    lr2, sig2 = projection.projection_schedule(40, initial_lr=0.2, initial_noise_factor=0.1)
    assert lr2[10] == pytest.approx(0.2 * (0.5 - 0.5 * math.cos(math.pi * min(1, 0.75 / 0.25))), rel=1e-14) and sig2[0] == 0.1


@pytest.mark.parametrize('delta', [1e-6, 1e-4])
def test_tolerance_basis_of_the_short_projections(delta):
    """Oracle against oracle with the VGG weights perturbed by `delta` (relative) at the `small` case of
    tests/test_gpu_projection.py (64 x 64, 3 modalities, B = 4, 40 steps): what a forward error of that size does to the
    final codes and the loss log.  The GPU tolerances in that file's header are derived from these numbers."""
    from oracle import lpips as olp
    from oracle import projector as opj
    G = _small()
    st = olp.random_vgg_state(7, TAPS)
    wa, ws = opj.w_stats(G)
    B, T = 4, 40
    y = _targets(G, B, 9, torch.float64)
    n = torch.randn([T, B, G.w_dim], generator=torch.Generator().manual_seed(4))
    w_ref, l_ref = opj.project(G, st, y, n.double(), w_avg=wa, w_std=ws, num_steps=T)
    g = torch.Generator().manual_seed(2)
    noisy = {k: v.double() * (1.0 + delta * torch.randn(v.shape, generator=g, dtype=torch.float64)) if k.startswith('features') else v
             for k, v in st.items()}
    w_p, l_p = opj.project(G, noisy, y, n.double(), w_avg=wa, w_std=ws, num_steps=T)
    ew = _rel(w_p, w_ref)
    el = float(((l_p - l_ref).abs() / l_ref.abs()).max())
    print(f'\nVGG weights perturbed by {delta:.0e}: final w rel-L2 {ew:.3e}, loss-log max rel {el:.3e}')
    # measured 3.3e-3 / 3.8e-4 (1e-6) and 5.1e-3 / 3.9e-4 (1e-4): even a 1e-6 perturbation moves w by a few 1e-3 (Adam
    # moves near-zero-gradient coordinates by +-lr on any last-bit difference).  The GPU tolerances (fp32_parity 1e-2 / 1e-3)
    # keep 1.5x or more above what the 1e-4 perturbation does.
    assert 1e-4 < ew < 1e-2 / 1.5 and el < 1e-3 / 1.5
    assert l_ref[-1] < l_ref[0]


class _StandInEngine:
    """What invert_dataset uses of a SynthesisEngine; the 'code' of an image is its mean pixel value, per batch row."""
    img_resolution, num_ws, w_dim = 8, 6, 16

    def __init__(self, batch):
        self.batch = batch
        self.targets = []
        self.calls = []

    def set_projection_targets(self, img):
        assert img.shape == (self.batch, 2, 8, 8) and img.dtype == torch.float32
        self.targets.append(img.clone())

    def project(self, num_steps, seed):
        self.calls.append((num_steps, seed))
        x = self.targets[-1]
        return x.mean((1, 2, 3)).reshape(-1, 1).repeat(1, self.w_dim) + torch.arange(self.w_dim) * 0.01


@pytest.mark.parametrize('batch', [4, 3])
def test_invert_dataset_writes_the_code_zip(tmp_path, batch):
    from latentaugment_b200.augments.utils import util_dataset as ud
    from latentaugment_b200.augments.utils import util_io
    src = os.path.join(os.path.dirname(__file__), 'golden', 'formats', 'images.zip')
    mods = ['MR_nonrigid_CT', 'MR_MR_T2']
    root = tmp_path / 'interim' / 'ds'
    root.mkdir(parents=True)
    out = root / 'codes.zip'
    eng = _StandInEngine(batch)
    n = util_io.invert_dataset(eng, src, str(out), split='train', modalities=mods, num_steps=7, seed=3)
    ds_i = ud.ImgDataset(src, 'train', mods, resolution=8)
    assert n == len(ds_i) == 16
    assert eng.calls == [(7, 3 + i) for i in range(math.ceil(16 / batch))]
    # inputs are x / 127.5 - 1, and the padded rows repeat the last image
    for bi, t in enumerate(eng.targets):
        rows = list(range(bi * batch, min(16, (bi + 1) * batch)))
        want = [ds_i[r][0] for r in rows] + [ds_i[rows[-1]][0]] * (batch - len(rows))
        assert torch.equal(t, torch.from_numpy(np.stack(want)) / 127.5 - 1)
    with zipfile.ZipFile(out) as z:
        assert sorted(z.namelist()) == ds_i.fnames
        w0 = pickle.loads(z.read(ds_i.fnames[0]))
    assert isinstance(w0, np.ndarray) and w0.dtype == np.float32 and w0.shape == (6, 16) and (w0 == w0[:1]).all()
    ds_w = ud.LatentCodeDataset(str(out), 'train', w_dim=16, num_ws=6)
    table = ds_w.to_table()
    names = ds_i.fnames[::3]
    want = torch.stack([torch.from_numpy(ds_i[ds_i.fnames.index(nm)][0]).mean() / 127.5 - 1 for nm in names])
    got = table.lookup(names).float().cpu()
    assert torch.allclose(got[:, 0], want.float(), atol=1e-6) and torch.allclose(got[:, 5] - got[:, 0], torch.full_like(want, 0.05).float(), atol=1e-6)
    # banks_from_reference_layout finds the zip under --interim_dir
    import shutil
    shutil.copy(src, root / 'imgs.zip')

    class Opt:
        interim_dir, dataset_aug, dataset_w_name, dataset_name_aug = str(tmp_path / 'interim'), 'ds', 'codes', 'imgs'
        modalities_aug, img_resolution, step_w, step_img = ','.join(mods), 8, 5, 10
    ds2, W, X = ud.banks_from_reference_layout(Opt, 'train', 16, 6)
    assert ds2.fnames == ds_i.fnames and W.shape[1:] == (6, 16) and 0 < W.shape[0] <= 16 and X.shape[1:] == (2, 8, 8)
    codes = torch.stack([torch.from_numpy(ds_w[i][0]) for i in range(len(ds_w))])
    assert all(bool((codes == row).all((1, 2)).any()) for row in W)         # the latent bank is made of the written codes


@pytest.mark.parametrize('win', [64, 128, 256])
def test_workspace_plans_the_target_features(win):
    """The per-sample target features take sum over taps of R^2 * C * 4 bytes per (sample, modality) -- ~32 MB at a 256
    window -- and only when asked for.  A 512 image projects through a 256 window, so it plans the same."""
    from latentaugment_b200 import _lib
    lib = _lib.load()
    d = _lib.VggDesc()
    for k in range(_lib.LA_VGG_TAPS):
        d.d_lin_weight[k] = 1024          # (planning reads only which taps are used)
    d.crop_size = win
    B, imgc = 32, 3
    sizes = {}
    for flag in (0, 1):
        d.per_sample_targets = flag
        n = C.c_size_t(0)
        _lib.check(lib.la_lpips_workspace_bytes(C.byref(d), B, imgc, _lib.PRECISION['bf16'], C.byref(n)))
        sizes[flag] = n.value
    per_crop = sum((win >> s) ** 2 * c * 4 for s, c in ((0, 64), (1, 128), (2, 256), (3, 512), (4, 512)))
    extra = sizes[1] - sizes[0]
    print(f'\nwindow {win}: target features {per_crop / 2**20:.1f} MB per crop, {extra / 2**30:.2f} GB at B = 32 x 3 modalities')
    assert B * imgc * per_crop <= extra <= B * imgc * per_crop + 5 * 1024
    if win == 256:
        assert 30 * 2**20 < per_crop < 32 * 2**20 and 2.8 < extra / 2**30 < 3.0


def test_invert_dataset_writes_several_splits_into_one_zip(tmp_path):
    from latentaugment_b200.augments.utils import util_dataset as ud
    from latentaugment_b200.augments.utils import util_io
    src = os.path.join(os.path.dirname(__file__), 'golden', 'formats', 'images.zip')
    mods = ['MR_nonrigid_CT', 'MR_MR_T2']
    out = tmp_path / 'codes.zip'
    eng = _StandInEngine(4)
    n = util_io.invert_dataset(eng, src, str(out), split=['train', 'val'], modalities=mods, num_steps=2, seed=0)
    assert n == 32 and [c[1] for c in eng.calls] == list(range(8))          # one seed per batch across the splits
    for sp in ('train', 'val'):
        assert ud.LatentCodeDataset(str(out), sp, w_dim=16, num_ws=6).fnames == ud.ImgDataset(src, sp, mods, resolution=8).fnames
