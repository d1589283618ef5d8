"""Optimisation core: B200-native counterpart of the reference
``augments/utils/util_latent_aug.py`` (``LatentAug``, ``define_latentaugment``).

The reference wraps one ``LatentAug`` nn.Module in ``nn.DataParallel`` (:20-33): every call
replicates G and the banks to each GPU, scatters ``w`` on dim 0 and runs an independent Adam
loop per replica with per-replica loss normalisers.  Here each GPU id owns one resident
``SynthesisEngine`` (weights and bank moments uploaded once); a call slices the batch the same
way and enqueues the replicas' loops asynchronously on their own devices -- same semantics,
no per-call replication.  For multi-process runs (one process per GPU, ``torchrun``) each
rank simply builds its own ``LatentAug`` over its batch shard (bench.py).
"""
import os
import random

import torch

from ... import engine as _engine
from . import util_dataset
from ...utils import synthetic
from ..criteria import create_criteria
from ..criteria.pix import center_crop_bounds


def l2_loss_vectorized(X, Y, compute_mean=True):
    """Pairwise squared L2, [bank, batch] orientation (reference :315-361) on the CUDA kernel."""
    if X.ndim not in (2, 3, 4) or Y.ndim != X.ndim:
        raise NotImplementedError
    D = _engine.pairwise_sqdist(X, Y)
    if compute_mean:
        D = D.sum() / (D.shape[0] * D.shape[1])
        n = 1
        for s in Y.shape[1:]:
            n *= s
        D = D / n
    return D


def get_crop_params(load_size, crop_size, preprocess='center_random_crop'):
    """Same two python ``random`` draws per call as the reference (util_dataset.py:284-296)."""
    new = load_size
    if preprocess == 'center_random_crop':
        new = center_crop_bounds(load_size)[1]
    x = random.randint(0, max(0, new - crop_size))
    y = random.randint(0, max(0, new - crop_size))
    return {'crop_pos': (x, y)}


def feature_bank_crops(X, res, crop_size, preprocess='center_random_crop'):
    """The windows the reference feeds to VGG when it builds ``fea_{mode}`` (compute_stats(manifold='features_*') ->
    extract_features_mode*, :564-598): for every modality, for every bank image, a FRESH ``get_params`` draw (two python
    ``random.randint`` calls) inside the centre crop.  X [M, C, res, res] -> [M, C, crop, crop]."""
    M, C = X.shape[0], X.shape[1]
    off = center_crop_bounds(res)[0] if preprocess == 'center_random_crop' else 0
    out = torch.empty([M, C, crop_size, crop_size], dtype=X.dtype)
    for c in range(C):
        for m in range(M):
            x, y = get_crop_params(res, crop_size, preprocess)['crop_pos']
            out[m, c] = X[m, c, off + y:off + y + crop_size, off + x:off + x + crop_size]
    return out


def reference_network_pickle_path(opt):
    """The reference's own location of the network pickle (``load_stylegan``, util_latent_aug.py:466-472):
    ``{model_dir}/{dataset_aug}/training-runs/{dataset_name_aug}/{modalities_aug}/<the one run whose name contains
    exp_stylegan>/{network_pkl_stylegan}``; ``None`` when ``--model_dir`` is unset or the tree does not exist."""
    model_dir = getattr(opt, 'model_dir', '')
    if not model_dir:
        return None
    dir_model = os.path.join(model_dir, opt.dataset_aug, 'training-runs', opt.dataset_name_aug, str(opt.modalities_aug))
    if not os.path.isdir(dir_model):
        return None
    runs = [x for x in os.listdir(dir_model) if opt.exp_stylegan in x]
    assert len(runs) == 1, f'{len(runs)} runs under {dir_model} match exp_stylegan={opt.exp_stylegan!r}: exactly one expected'
    return os.path.join(dir_model, runs[0], opt.network_pkl_stylegan)


def network_kwargs(nets):
    """The constructor arguments of a network pickle's modules that change what the engine computes, read from their
    ``init_kwargs`` (``torch_utils/persistence.py``): ``conv_clamp`` of G's synthesis network (``None`` for ``--cfg stylegan2``
    networks), ``disc_conv_clamp`` and ``mbstd_group_size`` of D (8 for the ``paper256`` / ``paper512`` configs).  Only the
    keys the pickle carries are returned; ``None`` means no clamp."""
    out = {}
    g_kw = getattr(nets.get('G_ema'), 'init_kwargs', None) or {}
    if 'conv_clamp' in (g_kw.get('synthesis_kwargs') or {}):
        out['conv_clamp'] = g_kw['synthesis_kwargs']['conv_clamp']
    d_kw = getattr(nets.get('D'), 'init_kwargs', None) or {}
    if 'conv_clamp' in d_kw:
        out['disc_conv_clamp'] = d_kw['conv_clamp']
    if 'mbstd_group_size' in (d_kw.get('epilogue_kwargs') or {}):
        out['mbstd_group_size'] = d_kw['epilogue_kwargs']['mbstd_group_size']
    return out


def load_stylegan_states(path):
    """``G_ema`` / ``D`` of a reference network pickle as plain ``state_dict``s (:473-484 keeps the modules; the engine reads
    parameters only), and the modules' constructor arguments the engine needs (``network_kwargs``).  The pickles embed the
    source of their classes and need the reference's ``torch_utils`` / ``dnnlib`` importable
    (``torch_utils/persistence.py:118-227``) -- true inside the reference's code base, which is where this plugin is dropped
    in; elsewhere convert once with ``tools/export_reference_pickle.py``.  Plain ``pickle.load`` as in the reference: only
    open files you trust."""
    import pickle
    print(f'Loading stylegan from "{path}"...')
    try:
        with open(path, 'rb') as f:
            nets = pickle.load(f)
    except ModuleNotFoundError as exc:
        raise ModuleNotFoundError(
            f'{exc}: the network pickle needs the reference\'s models/stylegan3 (torch_utils, dnnlib) on sys.path; or convert it '
            'once with tools/export_reference_pickle.py and pass --generator_state / --discriminator_state') from exc

    def sd(net):
        return {k: v.detach().cpu().float() for k, v in net.state_dict().items()}
    print('Done.')
    return sd(nets['G_ema']), (sd(nets['D']) if 'D' in nets else None), network_kwargs(nets)


class InvertedCodeTable:
    """Preloaded table of inverted codes keyed by sample file name: replaces the reference's
    per-sample zip read + unpickle in ``sample_from_inversion`` (latent_aug.py:310-324;
    SURVEY.md §8f rank 3) with one pinned ``[N, w_dim]`` tensor and an index lookup."""

    def __init__(self, names, codes):
        assert len(names) == codes.shape[0]
        self.index = {n: i for i, n in enumerate(names)}
        codes = codes.detach().float().reshape(len(names), -1).contiguous()
        self.codes = codes.pin_memory() if torch.cuda.is_available() else codes
        self._out = {}           # batch size -> two pinned staging buffers, used alternately

    def __len__(self):
        return self.codes.shape[0]

    def lookup(self, fnames):
        """[len(fnames), w_dim] gathered into a PINNED staging buffer (so the caller's ``.to(device, non_blocking=True)``
        really is asynchronous); two buffers per batch size alternate, so a result stays valid for one more call."""
        idx = torch.tensor([self.index[f] for f in fnames], dtype=torch.long)
        n = len(fnames)
        if n not in self._out:
            mk = (lambda: torch.empty([n, self.codes.shape[1]]).pin_memory()) if torch.cuda.is_available() else \
                (lambda: torch.empty([n, self.codes.shape[1]]))
            self._out[n] = [mk(), mk(), 0]
        slot = self._out[n]
        slot[2] ^= 1
        return torch.index_select(self.codes, 0, idx, out=slot[slot[2]])


class LatentAug:
    """Attributes mirror the reference class (:70-200): ``num_ws, w_dim, z_dim, batch_size,
    world_size, res, modalities, num_epochs, opt_lr, w_pix, w_lpips, w_latent, w_disc,
    soft_aug, alpha, truncation_psi, stats_dataset_w``; ``.module`` is the object itself (the
    reference reaches through ``DataParallel.module``, latent_aug.py:146-149,249)."""

    def __init__(self, phase, opt, save_dir, gpu_ids, generator_state=None, latent_bank=None, image_bank=None,
                 inverted_codes=None):
        if not gpu_ids:
            raise _engine._lib.LatentAugmentError('latentaugment_b200 has no CPU path: pass at least one GPU id')
        self.phase, self.opt, self.save_dir = phase, opt, save_dir
        self.gpu_ids = list(gpu_ids)
        self.world_size = len(self.gpu_ids)
        self.batch_size = opt.batch_size
        # micro-batches (addition): every GPU's shard is cut into k parts, each with its own engine, stream and captured graph,
        # all enqueued before any is awaited -- the latency-bound low-resolution launches of one part overlap the
        # tensor-core-bound launches of another and fill the tails of its persistent kernels.  Per-replica loss normalisers
        # stay those of the reference (n = batch / world): the term weights handed to a part are scaled by 1 / k.
        self.micro = max(1, int(getattr(opt, 'micro_batches', 1)))
        assert self.batch_size % (self.world_size * self.micro) == 0, 'batch_size must divide over gpu_ids_aug x micro_batches'
        self.num_epochs, self.opt_lr = opt.opt_num_epochs, opt.opt_lr
        self.w_pix, self.w_lpips, self.w_latent, self.w_disc = opt.w_pix, opt.w_lpips, opt.w_latent, opt.w_disc
        self.soft_aug, self.alpha = bool(opt.soft_aug), opt.alpha
        self.truncation_psi = opt.truncation_psi
        self.crop_size, self.preprocess = opt.crop_size_aug, opt.preprocess_aug
        self.verbose_flag = bool(getattr(opt, 'verbose_log', False))
        self.precision = getattr(opt, 'precision', 'fp32_parity')
        self.lpips_script = getattr(opt, 'lpips_script', 'lpips_script')
        self.criteria = create_criteria(opt)
        self.stats_loss, self.stats_time = {}, {}
        self.module = self

        # ---- generator (reference: load_stylegan, :466-484)
        pickle_disc_state, net_kw = None, {}
        if generator_state is None:
            pkl = None if getattr(opt, 'generator_state', '') else reference_network_pickle_path(opt)
            if getattr(opt, 'generator_state', ''):
                generator_state = torch.load(opt.generator_state, map_location='cpu', weights_only=True)
            elif pkl is not None:                                    # the reference's own --model_dir tree and pickle
                generator_state, pickle_disc_state, net_kw = load_stylegan_states(pkl)
            elif getattr(opt, 'synthetic', False):
                generator_state = synthetic.random_generator_state(
                    img_resolution=opt.img_resolution, img_channels=opt.synthetic_channels,
                    channel_base=opt.synthetic_channel_base, channel_max=opt.synthetic_channel_max, seed=0)
            else:
                raise FileNotFoundError(
                    'no generator given: pass --model_dir <the reference\'s tree holding its network pickle>, --generator_state '
                    '<state_dict.pt> (reference names, legacy.py:171-203) or --synthetic')
        self.generator_state = generator_state
        kw = synthetic.infer_generator_kwargs(generator_state)
        self.res, self.img_channels = kw['img_resolution'], kw['img_channels']
        self.w_dim, self.z_dim = kw['w_dim'], kw['z_dim']
        self.modalities = list(range(self.img_channels))
        # the pickle's own constructor arguments (None: no clamp); without a pickle the networks' defaults
        default_clamp = getattr(opt, 'conv_clamp', 256.0)
        conv_clamp = net_kw.get('conv_clamp', default_clamp)
        self.engines = []
        if self.micro > 1 and self.w_disc > 0:
            raise ValueError('--micro_batches > 1 changes the discriminator\'s minibatch-stddev groups: use 1 with w_disc > 0')
        for gid in self.gpu_ids:
            for _ in range(self.micro):
                self.engines.append(_engine.SynthesisEngine(
                    generator_state, batch=self.batch_size // (self.world_size * self.micro), precision=self.precision,
                    device=f'cuda:{gid}', conv_clamp=conv_clamp, **kw))
        self.num_ws = self.engines[0].num_ws
        self.device = self.engines[0].device

        # ---- banks (reference: compute_stats -> register_buffer('W' / 'X'), :140-158)
        gen = torch.Generator().manual_seed(1)
        if (latent_bank is None and image_bank is None and inverted_codes is None and getattr(opt, 'interim_dir', '')
                and not getattr(opt, 'latent_bank', '') and not getattr(opt, 'image_bank', '') and not getattr(opt, 'inverted_codes', '')):
            # the reference's own zips: {interim_dir}/{dataset_aug}/{dataset_w_name|dataset_name_aug}.zip (util_dataset.py)
            zpath = os.path.join(opt.interim_dir, opt.dataset_aug, opt.dataset_w_name + '.zip')
            if os.path.isfile(zpath):
                ds_w, latent_bank, image_bank = util_dataset.banks_from_reference_layout(
                    opt, phase, self.w_dim, self.num_ws, need_latent=self.w_latent > 0, need_img=self.w_pix > 0 or self.w_lpips > 0)
                inverted_codes = ds_w.to_table()
        if latent_bank is None and getattr(opt, 'latent_bank', ''):
            latent_bank = torch.load(opt.latent_bank, map_location='cpu', weights_only=True)
        if latent_bank is None and getattr(opt, 'synthetic', False):
            z = torch.randn([opt.synthetic_bank, self.z_dim], generator=gen)
            latent_bank = self.engines[0].mapping(z)[:, :1].cpu()
        if image_bank is None and getattr(opt, 'image_bank', ''):
            image_bank = torch.load(opt.image_bank, map_location='cpu', weights_only=True)
        if image_bank is None and getattr(opt, 'synthetic', False) and (self.w_pix > 0 or self.w_lpips > 0):
            image_bank = torch.rand([opt.synthetic_img_bank, self.img_channels, self.res, self.res],
                                    generator=torch.Generator().manual_seed(3)) * 2 - 1
        self.W = self.X = None
        if self.w_latent > 0:
            if latent_bank is None:
                raise FileNotFoundError('w_latent > 0 needs a latent bank (--latent_bank or --synthetic)')
            W = latent_bank.float()
            if W.ndim == 2:
                W = W.unsqueeze(1)
            if W.shape[1] == 1:
                W = W.repeat(1, self.num_ws, 1)
            self.W = W.to(self.device)
            for e in self.engines:
                self.criteria['latent'].attach(e, W)
        if self.w_pix > 0:
            if image_bank is None:
                raise FileNotFoundError('w_pix > 0 needs an image bank (--image_bank or --synthetic)')
            self.X = image_bank.float()
            for e in self.engines:
                self.criteria['pix'].attach(e, self.X)
        # ---- discriminator of the realism term (reference: self.D from the same pickle, :117)
        if self.w_disc > 0:
            disc_state, disc_kw = None, dict(conv_clamp=default_clamp)
            if getattr(opt, 'discriminator_state', ''):
                disc_state = torch.load(opt.discriminator_state, map_location='cpu', weights_only=True)
            elif pickle_disc_state is not None:                      # D of the same pickle, as the reference (:117)
                disc_state = pickle_disc_state
                disc_kw = dict(conv_clamp=net_kw.get('disc_conv_clamp', default_clamp), mbstd_group_size=net_kw.get('mbstd_group_size', 4))
            elif getattr(opt, 'synthetic', False):
                disc_state = synthetic.random_discriminator_state(
                    img_resolution=self.res, img_channels=self.img_channels, channel_base=opt.synthetic_channel_base,
                    channel_max=opt.synthetic_channel_max, seed=5)
            if disc_state is None:
                raise FileNotFoundError('w_disc > 0 needs a discriminator: --discriminator_state <state_dict.pt> '
                                        '(reference names, legacy.py:267-287) or --synthetic')
            for e in self.engines:
                self.criteria['disc'].attach(e, disc_state, **disc_kw)
        # ---- perceptual term (reference: self.vgg16 / self.lpips + register_buffer('fea_{mode}'), :125-131,160-181)
        if self.w_lpips > 0:
            vgg_state = None
            if getattr(opt, 'vgg_state', ''):
                vgg_state = torch.load(opt.vgg_state, map_location='cpu', weights_only=True)
            elif getattr(opt, 'synthetic', False):
                from ..criteria.lpips import taps_and_norm
                vgg_state = synthetic.random_vgg_state(seed=7, taps=taps_and_norm(self.lpips_script)[0])
            if vgg_state is None:
                raise FileNotFoundError('w_lpips > 0 needs the VGG16 + LPIPS parameters: --vgg_state <state_dict.pt> (torchvision '
                                        'features.* names + lin.{k}.weight) or --synthetic')
            if image_bank is None:
                raise FileNotFoundError('w_lpips > 0 needs an image bank (--image_bank or --synthetic)')
            self.X = image_bank.float() if self.X is None else self.X
            crops = feature_bank_crops(self.X, self.res, self.crop_size, self.preprocess)
            for e in self.engines:
                self.criteria['lpips'].attach(e, vgg_state, crops, lpips_script=self.lpips_script, crop_size=self.crop_size)
        # ---- inverted codes (reference: LatentCodeDataset zip, :140-143; latent_aug.py:310-324)
        if inverted_codes is None and getattr(opt, 'inverted_codes', ''):
            blob = torch.load(opt.inverted_codes, map_location='cpu', weights_only=True)      # {'names': [str], 'codes': tensor}
            inverted_codes = InvertedCodeTable(blob['names'], blob['codes'])
        if inverted_codes is None and getattr(opt, 'synthetic', False):
            n = opt.synthetic_codes
            z = torch.randn([n, self.z_dim], generator=torch.Generator().manual_seed(2))
            codes = torch.cat([self.engines[0].mapping(z[i:i + 256])[:, 0].cpu() for i in range(0, n, 256)])
            inverted_codes = InvertedCodeTable([f'synthetic_{i:05d}' for i in range(n)], codes)
        self.stats_dataset_w = inverted_codes

    # ---- reference helpers
    def broadcasting(self, latent):
        return latent.repeat([1, self.num_ws, 1])            # :493-494

    @staticmethod
    def reverse_broadcasting(latent):
        return latent[:, :1, :]                               # :496-498

    l2_loss_vectorized = staticmethod(l2_loss_vectorized)

    def calc_loss_latent(self, ws, W):
        return self.criteria['latent'](ws, W)

    def calc_loss_pix(self, x, x_bank):
        return self.criteria['pix'](x, x_bank)

    def calc_loss_lpips(self, x, crop_pos):
        """:387-424 (x is one engine's batch shard, uncropped; ``crop_pos`` from ``get_crop_params``)."""
        return self.criteria['lpips'](x, crop_pos)

    def calc_loss_disc(self, x):
        """:363-371 (x is one engine's batch shard)."""
        return self.criteria['disc'](x)

    def _shards(self, t):
        parts = self.world_size * self.micro
        n = self.batch_size // parts
        return [t[i * n:(i + 1) * n] for i in range(parts)]

    def z_to_w(self, z):
        """:459-464"""
        outs = [e.mapping(zs, truncation_psi=self.truncation_psi)[:, :1, :] for e, zs in zip(self.engines, self._shards(z))]
        return torch.cat([o.to(self.device) for o in outs])

    def forward_ganrand(self, z):
        """:202-205 -- G.mapping(z, None, truncation_psi) -> G.synthesis(w) (default noise mode)."""
        imgs, wss = [], []
        for e, zs in zip(self.engines, self._shards(z)):
            ws = e.mapping(zs, truncation_psi=self.truncation_psi)
            imgs.append(e.synthesis(ws, noise_mode='random'))
            wss.append(ws)
        return (torch.cat([i.to(self.device) for i in imgs]), torch.cat([w.to(self.device) for w in wss]))

    def forward(self, w, fname=None):
        """:207-310.  w [B, 1, w_dim] (or z [B, z_dim]) -> (img [B, C, res, res], w_aug [B, num_ws, w_dim])."""
        if w.ndim == 2:
            w = self.z_to_w(w)
        assert w.shape[0] == self.batch_size
        crop_pos = get_crop_params(self.res, self.crop_size, self.preprocess)['crop_pos']      # :216 (one window per call, feeds lpips)
        lpips_norm = self.criteria['lpips'].norm_mode if self.w_lpips > 0 else 0
        imgs, ws_out, self.last_losses = [], [], []
        k = 1.0 / self.micro            # a part's means run over batch / (world * micro) samples: rescale to the replica's normaliser
        for e, wsh in zip(self.engines, self._shards(w)):
            out = e.augment(wsh, num_steps=self.num_epochs, lr=self.opt_lr, w_latent=self.w_latent * k, w_pix=self.w_pix * k,
                            w_disc=self.w_disc, w_lpips=self.w_lpips * (k if lpips_norm == 0 else 1.0), lpips_crop=crop_pos,
                            lpips_norm_mode=lpips_norm, lpips_centre=self.preprocess == 'center_random_crop',
                            soft_aug=self.soft_aug, alpha=self.alpha, final_noise_mode='random',
                            return_losses=self.verbose_flag)
            imgs.append(out[0])
            ws_out.append(out[1])
            if self.verbose_flag:
                self.last_losses.append(out[2])
        img = torch.cat([i.to(self.device, non_blocking=True) for i in imgs]) if len(imgs) > 1 else imgs[0]
        w_aug = torch.cat([x.to(self.device, non_blocking=True) for x in ws_out]) if len(ws_out) > 1 else ws_out[0]
        if self.verbose_flag:
            self._log_first_call()
        return img, self.broadcasting(w_aug.unsqueeze(1))

    def _log_first_call(self):
        """Per-epoch loss values of the FIRST call only, as the reference logs them (:278-300: ``stats_loss[f'epoch_{t}']``,
        ``losses.jsonl`` in save_dir, then ``verbose_flag = False``); the matplotlib plots are not reproduced."""
        import json
        import os
        rows = (torch.stack([ll.cpu() for ll in self.last_losses]).sum(0) / self.world_size).tolist()   # parts summed, replicas averaged
        for t, row in enumerate(rows):
            self.stats_loss[f'epoch_{t}'] = {'loss_latent': row[0], 'loss_pix': row[1], 'loss_lpips': row[4], 'loss_disc': row[3], 'loss': row[2]}
            print(f'epoch {t + 1:>4d}/{self.num_epochs}, ' + ' '.join(f'{k} {v:<4.2f}' for k, v in self.stats_loss[f'epoch_{t}'].items()))
        if self.save_dir:
            try:
                os.makedirs(self.save_dir, exist_ok=True)
                with open(os.path.join(self.save_dir, 'losses.jsonl'), 'w') as f:
                    f.write(json.dumps(self.stats_loss, indent=2) + '\n')
            except OSError:
                pass
        self.verbose_flag = False

    __call__ = forward


def define_latentaugment(module_name, phase, opt, save_dir, gpu_ids, **kw):
    """:47-66"""
    if module_name == 'latent_aug':
        return LatentAug(phase, opt, save_dir, gpu_ids, **kw)
    raise NotImplementedError('LatentAugmentation module name [%s] is not recognized' % module_name)
