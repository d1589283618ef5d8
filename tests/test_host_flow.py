"""CPU tests of the plugin's HOST logic above the engine (``LatentAug`` / ``LatentAugment``): construction in synthetic
mode with all four criteria attached, sharding of a batch over ``--gpu_ids_aug 0,1`` x ``--micro_batches`` and the order the
parts come back in, the term-weight rescaling of micro-batches, the ``rand_aug`` path, the first-call loss log, the
look-ahead loop.  The CUDA engine is replaced by a recording stand-in (the engine itself is what the ``-m gpu`` tests
check); nothing here computes on a GPU."""
import json
import os

import pytest
import torch


class RecordingEngine:
    """Stands in for ``engine.SynthesisEngine``: same constructor and method signatures, arithmetic that makes the
    sample order visible (image i is filled with ``w0[i, 0, 0]``, ``w_aug = w0 + 1``)."""
    instances = []
    num_ws_of = staticmethod(lambda res: 2 * (res.bit_length() - 1) - 2)

    def __init__(self, state, *, img_resolution, img_channels, w_dim=512, z_dim=512, conv_clamp=256.0, batch, precision='fp32_parity',
                 device=None, mapping_lr_multiplier=0.01):
        self.res, self.C, self.w_dim, self.z_dim, self.batch, self.precision = img_resolution, img_channels, w_dim, z_dim, batch, precision
        self.requested_device = device
        self.device = torch.device('cpu')
        self.num_ws = type(self).num_ws_of(img_resolution)
        self.calls, self.launch_count = [], 0
        RecordingEngine.instances.append(self)

    def set_latent_bank(self, W):
        self.calls.append(('latent_bank', tuple(W.shape)))

    def set_image_bank(self, X):
        self.calls.append(('image_bank', tuple(X.shape)))

    def set_discriminator(self, state, channels=None, conv_clamp=256.0, mbstd_group_size=4):
        self.calls.append(('disc', len(state)))

    def set_lpips(self, state, taps=(16, 23, 30), crop_size=64, **kw):
        self.calls.append(('lpips', tuple(taps), crop_size))

    def set_feature_bank(self, crops):
        self.calls.append(('feature_bank', tuple(crops.shape)))

    def mapping(self, z, truncation_psi=1.0):
        return (z[:, :1, None] * truncation_psi).expand(z.shape[0], self.num_ws, self.w_dim).contiguous()

    def synthesis(self, ws, noise_mode='random', noise=None):
        self.calls.append(('synthesis', noise_mode, ws.shape[0]))
        return ws[:, 0, 0].reshape(-1, 1, 1, 1).expand(ws.shape[0], self.C, self.res, self.res).contiguous()

    def augment(self, w0, *, num_steps=10, lr=0.01, return_losses=False, **kw):
        assert w0.shape == (self.batch, 1, self.w_dim)
        self.calls.append(('augment', dict(kw, num_steps=num_steps, lr=lr)))
        img = w0[:, 0, 0].reshape(-1, 1, 1, 1).expand(self.batch, self.C, self.res, self.res).contiguous()
        out = (img, w0[:, 0] + 1.0)
        if return_losses:
            out += (torch.arange(num_steps * 5, dtype=torch.float32).reshape(num_steps, 5),)
        return out


@pytest.fixture
def fake_engine(monkeypatch):
    from latentaugment_b200 import engine
    RecordingEngine.instances = []
    monkeypatch.setattr(engine, 'SynthesisEngine', RecordingEngine)
    return RecordingEngine


def _make(argv, args, tmp_path=None):
    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.options.aug_options import AugOptions
    base = ['--aug', 'latent', '--synthetic', '--img_resolution', '128', '--synthetic_channels', '2', '--synthetic_channel_base', '8192',
            '--synthetic_channel_max', '64', '--synthetic_bank', '16', '--synthetic_img_bank', '5', '--synthetic_codes', '32']
    if tmp_path is not None:
        base += ['--checkpoints_dir', str(tmp_path)]
    opt = AugOptions().parse(args=dict({'p_thres': 0.0, 'init_w': 'inv'}, **args), argv=base + argv)
    aug = create_augment(opt)
    aug.device = torch.device('cpu')          # the caller-side device of the stand-in run
    aug._sync_forward = False
    return aug, opt


def _batch(aug, n, start=0):
    names = list(aug.stats_dataset_w.index)[start:start + n]
    return {'A': torch.zeros(n, 1, 128, 128), 'B': torch.zeros(n, 1, 128, 128), 'A_paths': names, 'B_paths': names}


def test_all_four_criteria_attach_and_batch_order_over_two_gpus_and_micro_batches(fake_engine):
    aug, opt = _make(['--batch_size', '8', '--gpu_ids_aug', '0,1', '--micro_batches', '2', '--opt_num_epochs', '3', '--no_log'],
                     {'w_disc': 0.0, 'w_lpips': 2.0, 'w_pix': 0.5, 'w_latent': 0.25})
    engs = fake_engine.instances
    assert [e.requested_device for e in engs] == ['cuda:0', 'cuda:0', 'cuda:1', 'cuda:1'] and all(e.batch == 2 for e in engs)
    for e in engs:
        kinds = [c[0] for c in e.calls]
        assert kinds[:2] == ['latent_bank', 'image_bank'] and 'lpips' in kinds and 'feature_bank' in kinds
        assert ('lpips', (4, 9, 16, 23, 30), 64) in e.calls                      # --lpips_script default: the five-tap form
        assert ('feature_bank', (5, 2, 64, 64)) in e.calls
    data = _batch(aug, 8)
    aug.set_input(data)
    aug.forward()
    out = aug.get_output()
    core = aug.latent_aug.module
    w_in = aug.w_AB                                                               # [8, 1, w_dim] as sampled from the table
    assert torch.equal(w_in[:, 0], core.stats_dataset_w.codes[:8])
    # part p of engine p comes back in position p: images carry w0[i, 0, 0]
    assert torch.equal(out['A'][:, 0, 0, 0], w_in[:, 0, 0]) and torch.equal(out['B'][:, 0, 0, 0], w_in[:, 0, 0])
    assert aug.w_AB_aug.shape == (8, core.num_ws, core.w_dim) and torch.equal(aug.w_AB_aug[:, 3], w_in[:, 0] + 1.0)
    # micro-batches: a part's means run over batch / (world * micro) samples -> pair-MEAN terms get weight / micro
    kw = [c[1] for c in engs[0].calls if c[0] == 'augment'][0]
    assert kw['w_latent'] == pytest.approx(0.125) and kw['w_pix'] == pytest.approx(0.25) and kw['w_lpips'] == pytest.approx(1.0)
    assert kw['num_steps'] == 3 and kw['lpips_norm_mode'] == 0 and kw['final_noise_mode'] == 'random' and kw['soft_aug'] is False
    # every part got the SAME crop window (drawn once per forward call, util_latent_aug.py:216)
    crops = {tuple(c[1]['lpips_crop']) for e in engs for c in e.calls if c[0] == 'augment'}
    assert len(crops) == 1
    assert aug.get_latent_output()['w'].shape == (8, core.w_dim) and aug.get_latent_input()['paths'] == data['A_paths']


def test_discriminator_term_refuses_micro_batches(fake_engine):
    with pytest.raises(ValueError):
        _make(['--batch_size', '4', '--micro_batches', '2', '--no_log'], {'w_lpips': 0.0})        # w_disc stays at its default of 1


def test_rand_aug_path(fake_engine):
    aug, opt = _make(['--batch_size', '4', '--rand_aug', '--no_log'], {'truncation_psi': 0.5})
    e = fake_engine.instances[0]
    assert opt.w_pix == opt.w_lpips == opt.w_latent == opt.w_disc == 0.0 and opt.opt_num_epochs == 0
    assert not any(c[0] in ('image_bank', 'lpips', 'disc') for c in e.calls)
    torch.manual_seed(3)
    z = torch.randn([4, aug.z_dim])
    torch.manual_seed(3)
    aug.set_input(_batch(aug, 4))
    aug.forward()
    out = aug.get_output()
    assert ('synthesis', 'random', 4) in e.calls and not any(c[0] == 'augment' for c in e.calls)
    assert torch.allclose(out['A'][:, 0, 0, 0], z[:, 0] * 0.5)                  # G.mapping(z, truncation_psi) -> G.synthesis, :202-205
    assert aug.get_latent_output()['paths'] == ''


def test_first_call_loss_log_and_lookahead_loop(fake_engine, tmp_path):
    aug, opt = _make(['--batch_size', '4', '--opt_num_epochs', '2', '--verbose_log', 'true'], {'w_lpips': 0.0, 'w_disc': 0.0}, tmp_path)
    core = aug.latent_aug.module
    batches = [_batch(aug, 4, 4 * i) for i in range(3)]
    got = list(aug.iterate(iter(batches)))
    assert [d['A_paths'] for d, _ in got] == [b['A_paths'] for b in batches]
    for (d, o), b in zip(got, batches):
        idx = [core.stats_dataset_w.index[n] for n in b['A_paths']]
        assert torch.equal(o['A'][:, 0, 0, 0], core.stats_dataset_w.codes[idx][:, 0])
    # the per-epoch losses of the FIRST call only (reference :278-300), columns (latent, pix, total, disc, lpips)
    assert sorted(core.stats_loss) == ['epoch_0', 'epoch_1'] and core.verbose_flag is False
    assert core.stats_loss['epoch_1'] == {'loss_latent': 5.0, 'loss_pix': 6.0, 'loss_lpips': 9.0, 'loss_disc': 8.0, 'loss': 7.0}
    log = os.path.join(core.save_dir, 'losses.jsonl')
    assert json.load(open(log)) == core.stats_loss
    assert len(aug.stats_time) == 3


def test_constructor_reads_the_reference_directory_layout(fake_engine, tmp_path, monkeypatch):
    """``--interim_dir`` pointing at the reference's tree (util_latent_aug.py:133-181): the zips of tests/golden/formats go in as
    they are -- banks by the slice schedule, inverted codes into the pinned table -- and what reaches the engine is what the
    REFERENCE's own classes made of the same zips (expected.pt, oracle/make_golden_formats.py)."""
    import shutil

    from conftest import GOLDEN
    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.options.aug_options import AugOptions
    from latentaugment_b200.utils import synthetic
    F = os.path.join(GOLDEN, 'formats')
    expected = torch.load(os.path.join(F, 'expected.pt'), weights_only=True)
    root = tmp_path / 'interim' / 'Pelvis'
    os.makedirs(root)
    shutil.copy(os.path.join(F, 'codes.zip'), root / 'codes-w.zip')
    shutil.copy(os.path.join(F, 'images.zip'), root / 'imgs.zip')
    state = synthetic.random_generator_state(img_resolution=8, img_channels=2, w_dim=16, z_dim=16, channel_base=256, channel_max=32)
    torch.save(state, tmp_path / 'g.pt')
    monkeypatch.setattr(fake_engine, 'num_ws_of', staticmethod(lambda res: 6))      # the fixture zips hold [6, 16] codes
    seen = {}
    monkeypatch.setattr(fake_engine, 'set_latent_bank', lambda self, W: seen.__setitem__('W', W.clone()))
    monkeypatch.setattr(fake_engine, 'set_image_bank', lambda self, X: seen.__setitem__('X', X.clone()))
    argv = ['--aug', 'latent', '--batch_size', '2', '--no_log', '--generator_state', str(tmp_path / 'g.pt'), '--img_resolution', '8',
            '--interim_dir', str(tmp_path / 'interim'), '--dataset_aug', 'Pelvis', '--dataset_w_name', 'codes-w', '--dataset_name_aug', 'imgs',
            '--step_w', '5', '--step_img', '10', '--checkpoints_dir', str(tmp_path)]
    opt = AugOptions().parse(args={'p_thres': 0.0, 'init_w': 'inv', 'w_lpips': 0.0, 'w_disc': 0.0}, argv=argv)
    aug = create_augment(opt)
    assert torch.equal(seen['W'].cpu(), expected['latent_step5']) and torch.equal(seen['X'].cpu(), expected['img_step10'])
    assert list(aug.stats_dataset_w.index) == expected['fnames']
    names = [expected['fnames'][0], expected['fnames'][7]]
    w = aug.sample_from_inversion(names)
    assert w.shape == (2, 1, 16) and torch.equal(w[0, 0], expected['w0'][0])
    assert os.path.isfile(root / 'cache_dir' / 'latent-step_5-maxitems_16.pkl')


def test_caller_loop_with_async_writer_matches_the_sequential_calls(fake_engine, tmp_path):
    """``util_io.augment_dataset`` (look-ahead loop + asynchronous pickle writer) leaves the files of the reference's inner
    loop (backbone_latentaug.py:91-124): same names, same dict layouts, same values as set_input / forward / get_output /
    get_latent_* called in sequence."""
    import numpy as np

    from latentaugment_b200.augments.utils import util_io
    aug, opt = _make(['--batch_size', '4', '--opt_num_epochs', '2', '--no_log'], {'w_lpips': 0.0, 'w_disc': 0.0})
    batches = [_batch(aug, 4, 4 * i) for i in range(5)]
    seq = []
    for b in batches[:3]:
        aug.set_input(b)
        aug.forward()
        o = aug.get_output()
        li, lo = aug.get_latent_input(), aug.get_latent_output()
        # (copies: with the stand-in engine everything stays on the CPU, so these are views of the code table's two staging buffers)
        seq.append(({k: (v.clone() if torch.is_tensor(v) else v) for k, v in o.items()}, dict(li, w=li['w'].copy()), dict(lo, w=lo['w'].copy())))
    out = tmp_path / 'run'
    for d in ('img', 'latent', 'img_aug'):                 # no latent_aug directory: that file is skipped, as in the reference
        os.makedirs(out / d)
    n = util_io.augment_dataset(aug, batches, str(out), n_iter=3, verbose=False)
    assert n == 3
    assert sorted(os.listdir(out / 'img')) == ['img_0', 'img_1', 'img_2'] and sorted(os.listdir(out / 'latent')) == ['w_0', 'w_1', 'w_2']
    assert sorted(os.listdir(out / 'img_aug')) == ['img_aug_0', 'img_aug_1', 'img_aug_2'] and not os.path.exists(out / 'latent_aug')
    for i in range(3):
        data = util_io.read_pickle(out / 'img' / f'img_{i}')
        assert data['A_paths'] == batches[i]['A_paths'] and torch.equal(data['A'], batches[i]['A'])
        got = util_io.read_pickle(out / 'img_aug' / f'img_aug_{i}')
        assert sorted(got) == ['A', 'A_paths', 'B', 'B_paths'] and got['A_paths'] == seq[i][0]['A_paths']
        assert torch.equal(got['A'], seq[i][0]['A']) and torch.equal(got['B'], seq[i][0]['B']) and got['A'].shape == (4, 1, 128, 128)
        w = util_io.read_pickle(out / 'latent' / f'w_{i}')
        assert isinstance(w['w'], np.ndarray) and w['w'].shape == seq[i][1]['w'].shape and np.array_equal(w['w'], seq[i][1]['w'])
        assert w['paths'] == seq[i][1]['paths']
    # augmented codes through the loop == get_latent_output of the sequential calls
    lat = [(wi, wo) for _, _, wi, wo in aug.iterate(iter(batches[:3]), with_latents=True)]
    for i in range(3):
        assert np.array_equal(lat[i][1]['w'], seq[i][2]['w']) and lat[i][1]['w'].shape == (4, aug.w_dim)


def test_async_writer_reports_errors_and_bounds_its_queue(tmp_path):
    from latentaugment_b200.augments.utils import util_io
    w = util_io.AsyncPickleWriter(max_pending=2)
    x = torch.arange(6.0)
    w.submit({'x': x}, str(tmp_path / 'a'))
    x += 1                                               # the writer owns a copy: later changes of the staging buffer do not leak
    w.close()
    assert torch.equal(util_io.read_pickle(tmp_path / 'a')['x'], torch.arange(6.0)) and w.written == 1
    w = util_io.AsyncPickleWriter()
    w.submit({'x': 1}, str(tmp_path / 'no_such_dir' / 'b'))
    with pytest.raises(OSError):
        w.close()


def test_constructor_loads_the_reference_network_pickle_tree(fake_engine, tmp_path, monkeypatch):
    """``--model_dir`` laid out as the reference expects (``load_stylegan``, util_latent_aug.py:466-484): the one run directory
    matching ``--exp_stylegan`` holds a pickle of ``{'G_ema': module, 'D': module}``; G's parameters reach the engine, D's the
    realism term -- no separate state files."""
    import pickle

    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.options.aug_options import AugOptions
    from oracle import sg2, sg2_disc
    cfg = dict(img_resolution=16, img_channels=2, channel_base=512, channel_max=32)
    G = sg2.Generator(**cfg).eval()
    D = sg2_disc.make_discriminator(**cfg)
    run = tmp_path / 'models' / 'DS' / 'training-runs' / 'DSname' / 'm0,m1' / '00003-stylegan2-DS-gpus2'
    os.makedirs(run)
    os.makedirs(run.parent / '00004-other-run')
    with open(run / 'network-snapshot-005320.pkl', 'wb') as f:
        pickle.dump({'G_ema': G, 'D': D, 'G': G}, f)
    seen = {}
    monkeypatch.setattr(fake_engine, 'set_discriminator', lambda self, state, **kw: seen.__setitem__('D', state))
    real_init = fake_engine.__init__

    def init(self, state, **kw):
        seen['G'] = state
        real_init(self, state, **kw)
    monkeypatch.setattr(fake_engine, '__init__', init)
    argv = ['--aug', 'latent', '--batch_size', '2', '--no_log', '--model_dir', str(tmp_path / 'models'), '--dataset_aug', 'DS',
            '--dataset_name_aug', 'DSname', '--modalities_aug', 'm0,m1', '--img_resolution', '16', '--checkpoints_dir', str(tmp_path),
            '--synthetic', '--synthetic_bank', '8', '--synthetic_img_bank', '3', '--synthetic_codes', '8',
            '--synthetic_channel_base', '512', '--synthetic_channel_max', '32']       # (--synthetic only supplies the banks here)
    opt = AugOptions().parse(args={'p_thres': 0.0, 'init_w': 'inv', 'w_lpips': 0.0, 'w_disc': 1.0}, argv=argv)
    aug = create_augment(opt)
    gs = G.state_dict()
    assert seen['G'].keys() == gs.keys() and all(torch.equal(seen['G'][k], gs[k].float()) for k in gs)
    ds = D.state_dict()
    assert seen['D'].keys() == ds.keys() and all(torch.equal(seen['D'][k], ds[k].float()) for k in ds)
    assert aug.latent_aug.module.res == 16 and aug.latent_aug.module.img_channels == 2
    # two runs matching the experiment id: refuse, as the reference's assert does
    os.makedirs(run.parent / '00003-duplicate')
    with pytest.raises(AssertionError):
        create_augment(opt)


@pytest.mark.parametrize('with_kwargs', [True, False])
def test_network_pickle_constructor_arguments_reach_the_engine(fake_engine, tmp_path, monkeypatch, with_kwargs):
    """The pickled modules' own ``init_kwargs`` (``torch_utils/persistence.py``) decide the clamp and the minibatch-stddev
    group, as they do when the reference runs the unpickled modules: a ``--cfg stylegan2`` G (``conv_clamp=None``) and a
    ``paper256`` D (``mbstd_group_size=8``, ``conv_clamp=256``).  Modules without ``init_kwargs`` keep the defaults."""
    import pickle

    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.options.aug_options import AugOptions
    from oracle import sg2, sg2_disc
    cfg = dict(img_resolution=16, img_channels=2, channel_base=512, channel_max=32)
    G = sg2.Generator(**cfg).eval()
    D = sg2_disc.make_discriminator(**cfg)
    if with_kwargs:
        G.init_kwargs = dict(z_dim=512, c_dim=0, w_dim=512, img_resolution=16, img_channels=2, mapping_kwargs={},
                             synthesis_kwargs=dict(channel_base=512, channel_max=32, num_fp16_res=0, conv_clamp=None))
        D.init_kwargs = dict(c_dim=0, img_resolution=16, img_channels=2, channel_base=512, channel_max=32, num_fp16_res=0,
                             conv_clamp=256, block_kwargs={}, mapping_kwargs={}, epilogue_kwargs=dict(mbstd_group_size=8))
    run = tmp_path / 'models' / 'DS' / 'training-runs' / 'DSname' / 'm0,m1' / '00003-stylegan2-DS-gpus2'
    os.makedirs(run)
    with open(run / 'network-snapshot-005320.pkl', 'wb') as f:
        pickle.dump({'G_ema': G, 'D': D}, f)
    seen = {}
    monkeypatch.setattr(fake_engine, 'set_discriminator', lambda self, state, **kw: seen.__setitem__('D', kw))
    real_init = fake_engine.__init__

    def init(self, state, **kw):
        seen['G'] = kw
        real_init(self, state, **kw)
    monkeypatch.setattr(fake_engine, '__init__', init)
    argv = ['--aug', 'latent', '--batch_size', '8', '--no_log', '--model_dir', str(tmp_path / 'models'), '--dataset_aug', 'DS',
            '--dataset_name_aug', 'DSname', '--modalities_aug', 'm0,m1', '--img_resolution', '16', '--checkpoints_dir', str(tmp_path),
            '--synthetic', '--synthetic_bank', '8', '--synthetic_img_bank', '3', '--synthetic_codes', '8',
            '--synthetic_channel_base', '512', '--synthetic_channel_max', '32']
    opt = AugOptions().parse(args={'p_thres': 0.0, 'init_w': 'inv', 'w_lpips': 0.0, 'w_disc': 1.0}, argv=argv)
    create_augment(opt)
    if with_kwargs:
        assert 'conv_clamp' in seen['G'] and seen['G']['conv_clamp'] is None
        assert seen['D'] == dict(conv_clamp=256, mbstd_group_size=8)
    else:
        assert seen['G']['conv_clamp'] == 256.0
        assert seen['D'] == dict(conv_clamp=256.0, mbstd_group_size=4)
