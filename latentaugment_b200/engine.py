"""Python host over the C ABI: owns device memory (torch tensors) and streams, nothing else.

``SynthesisEngine`` wraps one ``la_engine`` (one generator at one batch size).
"""
import ctypes as C
import math

import torch

from . import _lib
from . import projection as _proj

_PARAM_ORDER_DOC = 'parameter names follow the reference contract models/stylegan3/legacy.py:171-203'


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def generator_state(G):
    """state_dict-like mapping name -> tensor from an nn.Module or a plain dict."""
    sd = G if isinstance(G, dict) else dict(G.state_dict())
    return {k: v for k, v in sd.items()}


class SynthesisEngine:
    """One generator + batch size on one GPU.

    ``state``: mapping with the reference parameter names (``synthesis.b{res}.conv0.weight``,
    ``...affine.weight``, ``...noise_const``, ``...noise_strength``, ``synthesis.b4.const``,
    ``synthesis.b{res}.torgb.*``, ``synthesis.b{res}.resample_filter`` or
    ``synthesis.b{res}.conv0.resample_filter``, ``mapping.fc{i}.*``, ``mapping.w_avg``).
    """

    def __init__(self, state, *, img_resolution, img_channels, w_dim=512, z_dim=512, conv_clamp=256.0,
                 batch, precision='fp32_parity', device=None, mapping_lr_multiplier=0.01):
        if not torch.cuda.is_available():
            raise _lib.LatentAugmentError('latentaugment_b200 needs a CUDA device (sm_100a); there is no CPU path')
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f'cuda:{torch.cuda.current_device()}')
        self.batch, self.precision = int(batch), precision
        self.img_resolution, self.img_channels, self.w_dim, self.z_dim = img_resolution, img_channels, w_dim, z_dim
        log2 = int(math.log2(img_resolution))
        self.num_blocks = log2 - 1
        self.num_ws = 2 * self.num_blocks
        self._keep = []          # tensors whose storage the engine reads in place

        def dev(name, default=None):
            t = state.get(name, default)
            if t is None:
                raise KeyError(f'generator parameter {name!r} missing')
            t = torch.as_tensor(t).detach().to(self.device, torch.float32).contiguous()
            self._keep.append(t)
            return t

        d = _lib.GeneratorDesc()
        d.img_resolution, d.img_channels, d.w_dim, d.z_dim = img_resolution, img_channels, w_dim, z_dim
        d.num_blocks = self.num_blocks
        d.conv_clamp = float(conv_clamp) if conv_clamp is not None else -1.0
        d.d_const = _ptr(dev('synthesis.b4.const'))
        f = state.get('synthesis.b4.resample_filter', state.get('synthesis.b8.conv0.resample_filter'))
        if f is None:
            f1 = torch.tensor([1., 3., 3., 1.])
            f = torch.outer(f1, f1) / 64.0
        d.d_resample_filter = _ptr(dev('__filter__', f))
        li = 0
        self.conv_res = []
        for b in range(self.num_blocks):
            res = 4 << b
            names = (['conv0'] if b > 0 else []) + ['conv1']
            for nm in names:
                p = f'synthesis.b{res}.{nm}.'
                w = dev(p + 'weight')
                if nm == 'conv1':
                    d.channels[b] = w.shape[0]
                cp = d.conv[li]
                cp.d_weight, cp.d_bias = _ptr(w), _ptr(dev(p + 'bias'))
                cp.d_noise_const = _ptr(dev(p + 'noise_const'))
                cp.noise_strength = float(torch.as_tensor(state[p + 'noise_strength']).item())
                cp.d_affine_weight, cp.d_affine_bias = _ptr(dev(p + 'affine.weight')), _ptr(dev(p + 'affine.bias'))
                self.conv_res.append(res)
                li += 1
            p = f'synthesis.b{res}.torgb.'
            tp = d.torgb[b]
            tp.d_weight, tp.d_bias = _ptr(dev(p + 'weight')), _ptr(dev(p + 'bias'))
            tp.d_affine_weight, tp.d_affine_bias = _ptr(dev(p + 'affine.weight')), _ptr(dev(p + 'affine.bias'))
        nmap = 0
        while f'mapping.fc{nmap}.weight' in state and nmap < _lib.LA_MAX_MAPPING:
            d.d_mapping_weight[nmap] = _ptr(dev(f'mapping.fc{nmap}.weight'))
            d.d_mapping_bias[nmap] = _ptr(dev(f'mapping.fc{nmap}.bias'))
            nmap += 1
        d.mapping_layers = nmap
        d.mapping_lr_multiplier = mapping_lr_multiplier
        d.d_w_avg = _ptr(dev('mapping.w_avg', torch.zeros(w_dim)))
        self.desc = d

        nbytes = C.c_size_t(0)
        prec = _lib.PRECISION[precision]
        _lib.check(self.lib.la_engine_workspace_bytes(C.byref(d), self.batch, prec, C.byref(nbytes)))
        self.workspace_bytes = nbytes.value
        self.workspace = torch.empty(nbytes.value + 1024, dtype=torch.uint8, device=self.device)
        base = (self.workspace.data_ptr() + 1023) // 1024 * 1024
        handle = C.c_void_p(0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_engine_create(C.byref(d), self.batch, prec, C.c_void_p(base), nbytes.value,
                                                 _stream_ptr(self.device), C.byref(handle)))
        self.handle = handle
        self.noise_floats = self.lib.la_noise_floats(self.handle)

    def __del__(self):
        h = getattr(self, 'handle', None)
        if h:
            self.lib.la_engine_destroy(h)
            self.handle = None

    # ---- banks
    def set_latent_bank(self, W):
        W = W.detach().to(self.device, torch.float32).contiguous()
        if W.ndim == 2:
            W = W.unsqueeze(1).repeat(1, self.num_ws, 1).contiguous()
        assert W.shape[1:] == (self.num_ws, self.w_dim), W.shape
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_set_latent_bank(self.handle, _ptr(W), W.shape[0], _stream_ptr(self.device)))
        torch.cuda.current_stream(self.device).synchronize()      # W may be freed by the caller afterwards

    def set_image_bank(self, X):
        X = X.detach().to(self.device, torch.float32).contiguous()
        assert X.shape[1:] == (self.img_channels, self.img_resolution, self.img_resolution), X.shape
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_set_image_bank(self.handle, _ptr(X), X.shape[0], _stream_ptr(self.device)))
        torch.cuda.current_stream(self.device).synchronize()

    # ---- discriminator of the realism term (reference self.D, util_latent_aug.py:117,363-371)
    def set_discriminator(self, state, channels=None, conv_clamp=256.0, mbstd_group_size=4):
        """``state``: mapping with the reference parameter names of the StyleGAN2 'resnet' discriminator
        (``b{res}.{fromrgb,conv0,conv1,skip}.{weight,bias}``, ``b4.{conv,fc,out}.{weight,bias}``,
        ``b{res}.conv1.resample_filter``; models/stylegan3/legacy.py:267-287)."""
        state = generator_state(state)
        res = self.img_resolution
        blocks = []
        r = res
        while r > 4:
            blocks.append(r)
            r //= 2
        keep = self._disc_keep = []

        def dev(name):
            t = state[name].detach().to(self.device, torch.float32).contiguous()
            keep.append(t)
            return t
        d = _lib.DiscDesc()
        d.img_resolution, d.img_channels, d.num_blocks = res, self.img_channels, len(blocks)
        d.conv_clamp = -1.0 if conv_clamp is None else float(conv_clamp)
        d.mbstd_group_size = int(mbstd_group_size)
        for i, r in enumerate(blocks):
            d.channels[i] = state[f'b{r}.conv0.weight'].shape[0]
            b = d.block[i]
            if i == 0:
                b.d_fromrgb_weight = _ptr(dev(f'b{r}.fromrgb.weight'))
                b.d_fromrgb_bias = _ptr(dev(f'b{r}.fromrgb.bias'))
            b.d_conv0_weight, b.d_conv0_bias = _ptr(dev(f'b{r}.conv0.weight')), _ptr(dev(f'b{r}.conv0.bias'))
            b.d_conv1_weight, b.d_conv1_bias = _ptr(dev(f'b{r}.conv1.weight')), _ptr(dev(f'b{r}.conv1.bias'))
            b.d_skip_weight = _ptr(dev(f'b{r}.skip.weight'))
        d.channels[len(blocks)] = state['b4.fc.weight'].shape[0]
        fname = f'b{blocks[0]}.conv1.resample_filter'
        filt = state[fname] if fname in state else torch.outer(torch.tensor([1., 3., 3., 1.]), torch.tensor([1., 3., 3., 1.])) / 64
        keep.append(filt.detach().to(self.device, torch.float32).contiguous())
        d.d_resample_filter = _ptr(keep[-1])
        d.d_b4_conv_weight, d.d_b4_conv_bias = _ptr(dev('b4.conv.weight')), _ptr(dev('b4.conv.bias'))
        d.d_b4_fc_weight, d.d_b4_fc_bias = _ptr(dev('b4.fc.weight')), _ptr(dev('b4.fc.bias'))
        d.d_b4_out_weight, d.d_b4_out_bias = _ptr(dev('b4.out.weight')), _ptr(dev('b4.out.bias'))
        nbytes = C.c_size_t(0)
        _lib.check(self.lib.la_disc_workspace_bytes(C.byref(d), self.batch, _lib.PRECISION[self.precision], C.byref(nbytes)))
        self.disc_workspace = torch.empty(nbytes.value + 1024, dtype=torch.uint8, device=self.device)
        base = (self.disc_workspace.data_ptr() + 1023) // 1024 * 1024
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_set_discriminator(self.handle, C.byref(d), C.c_void_p(base), nbytes.value, _stream_ptr(self.device)))
        torch.cuda.current_stream(self.device).synchronize()
        self.has_disc = True

    def disc_logits(self, img):
        """reference ``self.D(x, c=None)``: img [batch, C, res, res] -> logits [batch, 1]."""
        img = img.detach().to(self.device, torch.float32).contiguous()
        assert img.shape == (self.batch, self.img_channels, self.img_resolution, self.img_resolution), img.shape
        out = torch.empty([self.batch], device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_disc_logits(self.handle, _ptr(img), _ptr(out), _stream_ptr(self.device)))
        return out.unsqueeze(1)

    def disc_loss_grad(self, img, w_disc=1.0):
        """(w_disc * softplus(-D(img)).mean(), its gradient wrt img) -- reference calc_loss_disc + autograd."""
        img = img.detach().to(self.device, torch.float32).contiguous()
        loss = torch.empty([1], device=self.device)
        grad = torch.empty_like(img)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_disc_loss_grad(self.handle, _ptr(img), float(w_disc), _ptr(loss), _ptr(grad), _stream_ptr(self.device)))
        return loss[0], grad

    # ---- perceptual term (reference self.vgg16 / self.lpips + the feature banks fea_{mode}, util_latent_aug.py:125-131,160-181)
    VGG_CONV_IDX = (0, 2, 5, 7, 10, 12, 14, 17, 19, 21, 24, 26, 28)      # torchvision vgg16.features indices of the 13 convs
    VGG_TAP_LAYERS = (4, 9, 16, 23, 30)                                  # 1-based layer indices of networks.py:52-64
    VGG_TAP_CHANNELS = (64, 128, 256, 512, 512)

    def set_lpips(self, state, taps=(16, 23, 30), crop_size=64, mean=(-.030, -.088, -.188), std=(.458, .448, .450),
                  per_sample_targets=False):
        """``state``: torchvision names ``features.{i}.{weight,bias}`` + LPIPS lin layers ``lin.{k}.weight`` ([1, C, 1, 1] or
        [C]; k counts the used ``taps`` in order; criteria/lpips/networks.py:22-32).  ``taps``: 1-based layer indices as in
        ``VGG16.target_layers`` (networks.py:94).  ``per_sample_targets``: also plan the target features of the projection
        (``set_projection_targets``; needs ``crop_size == min(img_resolution, 256)``)."""
        keep = self._lpips_keep = []

        def dev(t):
            t = torch.as_tensor(t).detach().to(self.device, torch.float32).contiguous()
            keep.append(t)
            return t
        d = _lib.VggDesc()
        for j, i in enumerate(self.VGG_CONV_IDX):
            d.d_conv_weight[j] = _ptr(dev(state[f'features.{i}.weight']))
            d.d_conv_bias[j] = _ptr(dev(state[f'features.{i}.bias']))
        for k, t in enumerate(taps):
            slot = self.VGG_TAP_LAYERS.index(t)
            w = dev(state[f'lin.{k}.weight']).reshape(-1)
            assert w.numel() == self.VGG_TAP_CHANNELS[slot], (t, w.shape)
            keep.append(w)
            d.d_lin_weight[slot] = _ptr(w)
        for k in range(3):
            d.mean[k], d.std[k] = float(mean[k]), float(std[k])
        d.crop_size = int(crop_size)
        d.per_sample_targets = int(bool(per_sample_targets))
        nbytes = C.c_size_t(0)
        _lib.check(self.lib.la_lpips_workspace_bytes(C.byref(d), self.batch, self.img_channels, _lib.PRECISION[self.precision], C.byref(nbytes)))
        self.lpips_workspace = torch.empty(nbytes.value + 1024, dtype=torch.uint8, device=self.device)
        base = (self.lpips_workspace.data_ptr() + 1023) // 1024 * 1024
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_set_lpips(self.handle, C.byref(d), C.c_void_p(base), nbytes.value, _stream_ptr(self.device)))
        torch.cuda.current_stream(self.device).synchronize()
        self.lpips_taps, self.lpips_crop = tuple(taps), int(crop_size)

    def set_feature_bank(self, crops):
        """Real crops [M, C, crop, crop] in [-1, 1] (one window per real image, util_latent_aug.py:564-579): the engine keeps the
        bank moments of their normalised VGG activations."""
        crops = crops.detach().to(self.device, torch.float32).contiguous()
        assert crops.shape[1:] == (self.img_channels, self.lpips_crop, self.lpips_crop), crops.shape
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_set_feature_bank(self.handle, _ptr(crops), crops.shape[0], _stream_ptr(self.device)))
        torch.cuda.current_stream(self.device).synchronize()

    def _crop_origin(self, crop_pos, centre):
        """Absolute window origin: ``crop_pos`` is drawn inside the centre crop when ``preprocess == 'center_random_crop'``
        (util_dataset.py:284-309)."""
        off = 0
        if centre:
            size = int(math.sqrt(self.img_resolution * self.img_resolution / 2))
            off = int(round((self.img_resolution - size) / 2.0))
        return int(crop_pos[0]) + off, int(crop_pos[1]) + off

    def lpips_loss_grad(self, img, crop_pos, w_lpips=1.0, norm_mode=0, centre=True):
        """(loss, d loss / d img) of the perceptual term alone -- reference calc_loss_lpips_* + autograd.  ``crop_pos`` =
        ``(x, y)`` from util_dataset.get_params (inside the centre crop when ``centre``)."""
        img = img.detach().to(self.device, torch.float32).contiguous()
        crop_pos = self._crop_origin(crop_pos, centre)
        loss = torch.empty([1], device=self.device)
        grad = torch.empty_like(img)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_lpips_loss_grad(self.handle, _ptr(img), int(crop_pos[0]), int(crop_pos[1]), float(w_lpips), int(norm_mode),
                                                   _ptr(loss), _ptr(grad), _stream_ptr(self.device)))
        return loss[0], grad

    def lpips_tap(self, k):
        """Normalised activations of used tap k from the last perceptual-term evaluation: [batch * C, h, w, C_tap] (NHWC)."""
        n = C.c_size_t(0)
        _lib.check(self.lib.la_lpips_tap(self.handle, k, C.c_void_p(0), C.byref(n), _stream_ptr(self.device)))
        out = torch.empty([n.value], device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_lpips_tap(self.handle, k, _ptr(out), C.byref(n), _stream_ptr(self.device)))
        slot = self.VGG_TAP_LAYERS.index(self.lpips_taps[k])
        ch = self.VGG_TAP_CHANNELS[slot]
        hw = int(round((n.value // (self.batch * self.img_channels * ch)) ** 0.5))
        return out.reshape(self.batch * self.img_channels, hw, hw, ch)

    # ---- projection of real images into W (projector.py::project, batched; DESIGN.md "Projection")
    def set_projection_targets(self, img):
        """Targets [batch, C, res, res] in [-1, 1] (``x / 127.5 - 1`` of the 0..255 images).  Needs ``set_lpips(...,
        per_sample_targets=True)``."""
        img = img.detach().to(self.device, torch.float32).contiguous()
        assert img.shape == (self.batch, self.img_channels, self.img_resolution, self.img_resolution), img.shape
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_set_projection_targets(self.handle, _ptr(img), _stream_ptr(self.device)))
        torch.cuda.current_stream(self.device).synchronize()

    def projection_loss_grad(self, img):
        """(per-sample distance [batch] of ``img`` to the projection targets, d sum / d img): the projection's loss alone."""
        img = img.detach().to(self.device, torch.float32).contiguous()
        loss = torch.empty([self.batch], device=self.device)
        grad = torch.empty_like(img)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_lpips_loss_grad(self.handle, _ptr(img), 0, 0, 1.0, 2, _ptr(loss), _ptr(grad), _stream_ptr(self.device)))
        return loss, grad

    def w_stats(self):
        """(w_avg [w_dim], w_std) of 10 000 mapped ``z`` (``RandomState(123)``, psi = 1, row 0), float64 on the host; cached."""
        if getattr(self, '_w_stats', None) is None:
            if self.desc.mapping_layers < 1:
                raise _lib.LatentAugmentError('projection needs the mapping network (w_avg / w_std); this generator has none')
            z = torch.from_numpy(_proj.w_avg_z(self.z_dim)).float().to(self.device)
            w = torch.empty([z.shape[0], self.w_dim], device=self.device)
            with torch.cuda.device(self.device):
                for i in range(0, z.shape[0], self.batch):
                    j = min(z.shape[0], i + self.batch)
                    _lib.check(self.lib.la_mapping(self.handle, _ptr(z[i:j]), j - i, 1.0, _ptr(w[i:j]), _stream_ptr(self.device)))
            self._w_stats = _proj.w_stats_from_samples(w.cpu().double().numpy())
        return self._w_stats

    def project(self, w0=None, *, num_steps=_proj.NUM_STEPS, initial_lr=_proj.INITIAL_LR, initial_noise_factor=_proj.INITIAL_NOISE_FACTOR,
                lr_rampdown_length=_proj.LR_RAMPDOWN_LENGTH, lr_rampup_length=_proj.LR_RAMPUP_LENGTH,
                noise_ramp_length=_proj.NOISE_RAMP_LENGTH, w_noise=None, seed=0, return_losses=False):
        """Projects the targets of ``set_projection_targets`` into W: ``num_steps`` Adam steps on one code per sample from
        ``w0`` [batch, w_dim] (default ``w_avg``).  ``w_noise`` [T, batch, w_dim] unit normal draws of the w noise (default: drawn
        on the CPU from ``torch.Generator().manual_seed(seed)``).  Returns w [batch, w_dim] (and the summed loss of every step)."""
        T, B = int(num_steps), self.batch
        w_avg, w_std = self.w_stats()
        if w0 is None:
            w0 = torch.from_numpy(w_avg).float().unsqueeze(0).repeat(B, 1)
        w0 = w0.detach().to(self.device, torch.float32).reshape(B, self.w_dim).contiguous()
        lr, sigma = _proj.projection_schedule(T, initial_lr=initial_lr, initial_noise_factor=initial_noise_factor,
                                              lr_rampdown_length=lr_rampdown_length, lr_rampup_length=lr_rampup_length,
                                              noise_ramp_length=noise_ramp_length)
        lr = torch.from_numpy(lr).float().to(self.device)
        sigma = torch.from_numpy(sigma * w_std).float().to(self.device)
        if w_noise is None:
            w_noise = torch.randn([T, B, self.w_dim], generator=torch.Generator().manual_seed(int(seed)))
        w_noise = w_noise.detach().to(self.device, torch.float32).contiguous()
        assert w_noise.shape == (T, B, self.w_dim), w_noise.shape
        w = torch.empty([B, self.w_dim], device=self.device)
        losses = torch.zeros([max(T, 1)], device=self.device) if return_losses else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_project(self.handle, _ptr(w0), T, _ptr(lr), _ptr(sigma), _ptr(w_noise), _ptr(w), _ptr(losses),
                                           _stream_ptr(self.device)))
        if return_losses:
            return w, losses[:T]
        return w

    # ---- network
    def mapping(self, z, truncation_psi=1.0):
        """[n, z_dim] -> [n, num_ws, w_dim] (broadcast rows), reference G.mapping(z, None, truncation_psi)."""
        z = z.detach().to(self.device, torch.float32).contiguous()
        n = z.shape[0]
        out = torch.empty([n, self.w_dim], device=self.device)
        with torch.cuda.device(self.device):
            for i in range(0, n, self.batch):
                j = min(n, i + self.batch)
                _lib.check(self.lib.la_mapping(self.handle, _ptr(z[i:j]), j - i, float(truncation_psi), _ptr(out[i:j]),
                                               _stream_ptr(self.device)))
        return out.unsqueeze(1).repeat(1, self.num_ws, 1)

    def _noise(self, noise_mode, noise):
        if noise_mode != 'random':
            return None
        if noise is None:
            noise = torch.randn([self.noise_floats], device=self.device)
        elif isinstance(noise, (list, tuple)):
            noise = torch.cat([n.reshape(-1) for n in noise])
        noise = noise.detach().to(self.device, torch.float32).contiguous()
        assert noise.numel() == self.noise_floats, (noise.numel(), self.noise_floats)
        return noise

    def synthesis(self, ws, noise_mode='random', noise=None):
        """reference G.synthesis(ws, noise_mode=...): ws [batch, num_ws, w_dim] -> [batch, C, res, res]."""
        ws = ws.detach().to(self.device, torch.float32).contiguous()
        assert ws.shape == (self.batch, self.num_ws, self.w_dim), ws.shape
        nz = self._noise(noise_mode, noise)
        img = torch.empty([self.batch, self.img_channels, self.img_resolution, self.img_resolution], device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_synthesis(self.handle, _ptr(ws), self.num_ws * self.w_dim, self.w_dim,
                                             _lib.NOISE[noise_mode], _ptr(nz), _ptr(img), _stream_ptr(self.device)))
        return img

    def augment(self, w0, *, num_steps=10, lr=0.01, w_latent=1.0, w_pix=1.0, w_disc=0.0, w_lpips=0.0, lpips_crop=(0, 0),
                lpips_norm_mode=0, lpips_centre=True, soft_aug=False, alpha=1.0, final_noise_mode='random', final_noise=None,
                return_losses=False):
        """The hot path (reference LatentAug.forward).  w0 [batch, w_dim] or [batch, 1, w_dim]."""
        w0 = w0.detach().to(self.device, torch.float32).reshape(self.batch, self.w_dim).contiguous()
        nz = self._noise(final_noise_mode, final_noise)
        img = torch.empty([self.batch, self.img_channels, self.img_resolution, self.img_resolution], device=self.device)
        w_aug = torch.empty([self.batch, self.w_dim], device=self.device)
        lpips_crop = self._crop_origin(lpips_crop, lpips_centre) if w_lpips > 0 else (0, 0)
        nlog = min(max(num_steps, 1), _lib.LA_MAX_STEPS)
        losses = torch.zeros([nlog, _lib.LA_LOSS_COLS], device=self.device) if return_losses else None
        opt = _lib.AugmentOptions(num_steps, lr, w_latent, w_pix, int(bool(soft_aug)), alpha, _lib.NOISE[final_noise_mode],
                                  self.img_channels, w_disc, w_lpips, int(lpips_crop[0]), int(lpips_crop[1]), int(lpips_norm_mode))
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_augment(self.handle, _ptr(w0), C.byref(opt), _ptr(nz), _ptr(img), _ptr(w_aug), _ptr(losses),
                                           _stream_ptr(self.device)))
        if return_losses:
            return img, w_aug, losses[:min(num_steps, nlog)]      # columns: latent, pixel, total, discriminator, perceptual
        return img, w_aug

    # ---- debug hooks (tests)
    def debug_set_simt(self, flag):
        _lib.check(self.lib.la_debug_set_simt(self.handle, int(flag)))

    def debug_check(self):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_debug_check(self.handle, _stream_ptr(self.device)))

    def debug_get(self, what):
        """Internal quantity of the last optimisation step (``la_debug_get``): 'g_s' | 's' | 'd' | 'grad_w' | 'soff'."""
        code = {'g_s': 0, 's': 1, 'd': 2, 'grad_w': 3, 'soff': 4}[what]
        n = C.c_size_t(0)
        _lib.check(self.lib.la_debug_get(self.handle, code, C.c_void_p(0), C.byref(n), _stream_ptr(self.device)))
        out = torch.empty([n.value], device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_debug_get(self.handle, code, _ptr(out), C.byref(n), _stream_ptr(self.device)))
        return out

    def debug_time_gemms(self, reps=5):
        """Per-launch device time (ms) of every tap-GEMM of one optimisation step, timed alone."""
        n = len(self.conv_res)
        buf = (C.c_float * (4 * n + 1))()
        nl = C.c_int(0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_debug_time_gemms(self.handle, reps, buf, C.byref(nl)))
        assert nl.value == n
        v = list(buf)
        return {'forward': v[:n], 'dgrad': v[n:2 * n], 'fir_forward': v[2 * n:3 * n], 'fir_backward': v[3 * n:4 * n], 'seed': v[4 * n]}

    @property
    def launch_count(self):
        return self.lib.la_debug_launch_count(self.handle)


def pairwise_sqdist(X, Y):
    """D [m, n] = l2_loss_vectorized(X, Y, compute_mean=False) (reference util_latent_aug.py:315-361)."""
    lib = _lib.load()
    n, m = X.shape[0], Y.shape[0]
    X = X.detach().reshape(n, -1).float().contiguous()
    Y = Y.detach().reshape(m, -1).float().contiguous()
    D = torch.empty([m, n], device=X.device)
    with torch.cuda.device(X.device):
        _lib.check(lib.la_pairwise_sqdist(_ptr(X), n, _ptr(Y), m, X.shape[1], _ptr(D), _stream_ptr(X.device)))
    return D


class LatentBank:
    """Device-resident real-code bank (or one shard of it) prepared for nearest-code queries."""

    def __init__(self, Y, index_offset=0):
        self.lib = _lib.load()
        m = Y.shape[0]
        self.Y = Y.detach().reshape(m, -1).float().contiguous()
        self.m, self.K = m, self.Y.shape[1]
        self.index_offset = int(index_offset)
        self.bf16 = torch.empty([m, self.K], dtype=torch.bfloat16, device=self.Y.device)
        self.sqnorm = torch.empty([m + 1], device=self.Y.device)          # |y_j|^2 followed by their maximum
        with torch.cuda.device(self.Y.device):
            _lib.check(self.lib.la_bank_prepare(_ptr(self.Y), m, self.K, _ptr(self.bf16), _ptr(self.sqnorm),
                                                _stream_ptr(self.Y.device)))
        self._ws = None

    def nearest(self, X, k=1, out=None):
        """(dist [n, k], idx [n, k] int64) of the k nearest bank rows per query, ties to the lowest index.
        ``out = (dist, idx)``: preallocated contiguous result tensors (graph-captured callers)."""
        n = X.shape[0]
        X = X.detach().reshape(n, -1).float().contiguous()
        assert X.shape[1] == self.K
        nbytes = C.c_size_t(0)
        _lib.check(self.lib.la_nearest_codes_workspace_bytes(n, self.m, self.K, k, C.byref(nbytes)))
        if self._ws is None or self._ws.numel() < nbytes.value + 1024:
            self._ws = torch.empty(nbytes.value + 1024, dtype=torch.uint8, device=X.device)
        base = (self._ws.data_ptr() + 1023) // 1024 * 1024
        if out is None:
            dist = torch.empty([n, k], device=X.device)
            idx = torch.empty([n, k], dtype=torch.int64, device=X.device)
        else:
            dist, idx = out
            assert dist.is_contiguous() and idx.is_contiguous() and dist.shape == (n, k) and idx.shape == (n, k)
        with torch.cuda.device(X.device):
            _lib.check(self.lib.la_nearest_codes(_ptr(X), n, _ptr(self.Y), _ptr(self.bf16), _ptr(self.sqnorm), self.m, self.K,
                                                 k, self.index_offset, C.c_void_p(base), nbytes.value, _ptr(dist), _ptr(idx),
                                                 _stream_ptr(X.device)))
        return dist, idx


class FeatureManifold:
    """Device-resident feature manifold of the precision / recall metric (DESIGN.md §12): the features rounded to fp16
    (held as fp32), their hi | lo bf16 planes and squared norms.  ``fallback`` is a device int32 counter to which every
    call adds the queries that were scanned exhaustively."""

    ROWS_PER_CALL = 8192          # bounds the per-call workspace (candidate lists, query planes): ~0.2 GB at 50 000 x 4096

    def __init__(self, Y):
        self.lib = _lib.load()
        m = Y.shape[0]
        self.Y = Y.detach().reshape(m, -1).to(torch.float16).float().contiguous()
        self.m, self.K = m, self.Y.shape[1]
        dev = self.Y.device
        self.planes = torch.empty([2, m, self.K], dtype=torch.bfloat16, device=dev)
        self.sqnorm = torch.empty([m + 1], device=dev)
        self.fallback = torch.zeros([1], dtype=torch.int32, device=dev)
        self._ws = None
        with torch.cuda.device(dev):
            _lib.check(self.lib.la_pr_manifold_prepare(_ptr(self.Y), m, self.K, _ptr(self.planes), _ptr(self.sqnorm), _stream_ptr(dev)))

    def _workspace(self, nbytes):
        if self._ws is None or self._ws.numel() < nbytes + 1024:
            self._ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.Y.device)
        return C.c_void_p((self._ws.data_ptr() + 1023) // 1024 * 1024)

    def radii(self, begin=0, end=None, nhood_size=3):
        """r2 [end - begin]: the (nhood+1)-th smallest squared distance of manifold rows [begin, end) over the manifold."""
        end = self.m if end is None else end
        dev = self.Y.device
        r2 = torch.empty([end - begin], device=dev)
        with torch.cuda.device(dev):
            for b in range(begin, end, self.ROWS_PER_CALL):
                n = min(self.ROWS_PER_CALL, end - b)
                nbytes = C.c_size_t(0)
                _lib.check(self.lib.la_pr_radii_workspace_bytes(n, self.m, self.K, nhood_size, C.byref(nbytes)))
                ws = self._workspace(nbytes.value)
                _lib.check(self.lib.la_pr_radii(C.c_void_p(self.Y.data_ptr() + b * self.K * 4), n, _ptr(self.Y), _ptr(self.planes),
                                                _ptr(self.sqnorm), self.m, self.K, nhood_size, ws, nbytes.value,
                                                C.c_void_p(r2.data_ptr() + (b - begin) * 4), _ptr(self.fallback), _stream_ptr(dev)))
        return r2

    def member(self, X, r2):
        """uint8 [n]: 1 where probe i lies in some manifold ball, h(d2(x_i, y_j)) <= h(r2_j); r2 [m] from ``radii``."""
        n = X.shape[0]
        X = X.detach().reshape(n, -1).to(torch.float16).float().contiguous()
        r2 = r2.float().contiguous()
        assert X.shape[1] == self.K and r2.shape == (self.m,)
        dev = self.Y.device
        out = torch.empty([n], dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            for b in range(0, n, self.ROWS_PER_CALL):
                c = min(self.ROWS_PER_CALL, n - b)
                nbytes = C.c_size_t(0)
                _lib.check(self.lib.la_pr_member_workspace_bytes(c, self.m, self.K, C.byref(nbytes)))
                ws = self._workspace(nbytes.value)
                _lib.check(self.lib.la_pr_member(C.c_void_p(X.data_ptr() + b * self.K * 4), c, _ptr(self.Y), _ptr(self.planes),
                                                 _ptr(self.sqnorm), _ptr(r2), self.m, self.K, ws, nbytes.value,
                                                 C.c_void_p(out.data_ptr() + b), _ptr(self.fallback), _stream_ptr(dev)))
        return out


IMAGENET_MEAN = tuple(255.0 * v for v in (0.485, 0.456, 0.406))     # torchvision's normalisation, in the 0..255 domain
IMAGENET_STD = tuple(255.0 * v for v in (0.229, 0.224, 0.225))


class FeatureDetector:
    """VGG16 detector of precision / recall (DESIGN.md §13): torchvision ``vgg16`` up to the ReLU of fc7 on the GPU.

    ``state``: torchvision names ``features.{i}.{weight,bias}`` and ``classifier.{0,3}.{weight,bias}`` (e.g.
    ``torchvision.models.vgg16(...).state_dict()``).  ``batch``: images per call of the native detector (its workspace is
    planned for that many); ``features`` walks any number of images in chunks of ``batch``.  ``mean`` / ``std``: per-channel
    normalisation of the 0..255 input (default torchvision's ImageNet constants x 255)."""

    VGG_CONV_IDX = SynthesisEngine.VGG_CONV_IDX
    DIM = 4096

    def __init__(self, state, batch=256, precision='bf16', mean=IMAGENET_MEAN, std=IMAGENET_STD, device=None):
        self.lib = _lib.load()
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        self.batch, self.precision = int(batch), precision
        keep = self._params = []

        def dev(t):
            t = torch.as_tensor(t).detach().to(self.device, torch.float32).contiguous()
            keep.append(t)
            return _ptr(t)
        d = _lib.DetectorDesc()
        for j, i in enumerate(self.VGG_CONV_IDX):
            d.d_conv_weight[j] = dev(state[f'features.{i}.weight'])
            d.d_conv_bias[j] = dev(state[f'features.{i}.bias'])
        assert tuple(state['classifier.0.weight'].shape) == (4096, 25088) and tuple(state['classifier.3.weight'].shape) == (4096, 4096)
        d.d_fc6_weight, d.d_fc6_bias = dev(state['classifier.0.weight']), dev(state['classifier.0.bias'])
        d.d_fc7_weight, d.d_fc7_bias = dev(state['classifier.3.weight']), dev(state['classifier.3.bias'])
        for k in range(3):
            d.mean[k], d.std[k] = float(mean[k]), float(std[k])
        prec = _lib.PRECISION[precision]
        nbytes = C.c_size_t(0)
        _lib.check(self.lib.la_detector_workspace_bytes(C.byref(d), self.batch, prec, C.byref(nbytes)))
        self.workspace = torch.empty(nbytes.value + 1024, dtype=torch.uint8, device=self.device)
        base = (self.workspace.data_ptr() + 1023) // 1024 * 1024
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.la_detector_create(C.byref(d), self.batch, prec, C.c_void_p(base), nbytes.value, _stream_ptr(self.device),
                                                   C.byref(h)))
        self.handle = h
        # only the biases are read in place; the prepared operands of the weights live in the workspace
        self._params = [t for t in keep if t.dim() == 1]

    def __del__(self):
        h = getattr(self, 'handle', None)
        if h:
            torch.cuda.synchronize(self.device)
            self.lib.la_detector_destroy(h)
            self.handle = None

    def features(self, img, modality=0):
        """fp32 [n, 4096] on the detector's GPU: fc7 embeddings of channel ``modality`` of ``img`` [n, C, H, W] (H == W,
        values in [-1, 1], on any device)."""
        n, c, hh, ww = img.shape
        assert hh == ww, img.shape
        out = torch.empty([n, self.DIM], device=self.device)
        with torch.cuda.device(self.device):
            for b in range(0, n, self.batch):
                e = min(n, b + self.batch)
                x = img[b:e].detach().to(self.device, torch.float32).contiguous()
                _lib.check(self.lib.la_detector_features(self.handle, _ptr(x), e - b, c, hh, int(modality), _ptr(out[b:e]),
                                                         _stream_ptr(self.device)))
        return out


def merge_topk(dist, idx):
    """[shards, n, k] -> [n, k] global k best (ties to the lowest index)."""
    lib = _lib.load()
    s, n, k = dist.shape
    dist = dist.float().contiguous()
    idx = idx.to(torch.int64).contiguous()
    od = torch.empty([n, k], device=dist.device)
    oi = torch.empty([n, k], dtype=torch.int64, device=dist.device)
    with torch.cuda.device(dist.device):
        _lib.check(lib.la_merge_topk(_ptr(dist), _ptr(idx), s, n, k, _ptr(od), _ptr(oi), _stream_ptr(dist.device)))
    return od, oi
