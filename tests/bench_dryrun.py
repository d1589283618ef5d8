"""CPU dry run of bench.py's CONTROL FLOW (not a measurement): the CUDA-facing pieces are replaced by small torch-CPU
stand-ins so that the whole default run -- headline legs, the C5 / C3 extra legs, the one-line emitter, the watchdogs and
the process-group teardown -- executes here, single process or under a world-size-2 ``gloo`` group.  Launched by
tests/test_bench_flow.py as ``python tests/bench_dryrun.py [bench.py flags]`` with RANK / WORLD_SIZE / MASTER_* set.
"""
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch
import torch.distributed as dist

import bench

HANG = os.environ.get('DRYRUN_HANG', '')           # 'c5': the C5 leg never returns on rank 0; 'teardown': destroy hangs


class _Event:
    def __init__(self, enable_timing=False):
        self.t = 0.0

    def record(self):
        import time
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-3)


_real_device = torch.device
_cpu = _real_device('cpu')


class _Dev:
    """stands in for torch.device('cuda:i'): tensors stay on the CPU, ``index`` is kept"""

    def __init__(self, index):
        self.index = index


_real_to = torch.Tensor.to


def _to(self, *a, **k):
    a = tuple(_cpu if isinstance(x, _Dev) else x for x in a)
    k = {n: (_cpu if isinstance(v, _Dev) else v) for n, v in k.items()}
    k.pop('non_blocking', None)
    return _real_to(self, *a, **k)


_real_tensor = torch.tensor
_real_empty = torch.empty


def _strip_dev(fn):
    def wrapped(*a, **k):
        if isinstance(k.get('device'), _Dev):
            k['device'] = _cpu
        return fn(*a, **k)
    return wrapped


def patch_torch():
    torch.cuda.set_device = lambda *_: None
    torch.cuda.synchronize = lambda *_: None
    torch.cuda.empty_cache = lambda: None
    torch.cuda.Event = _Event
    bench.cuda_device = _Dev
    torch.Tensor.to = _to
    torch.Tensor.pin_memory = lambda self: self
    torch.tensor = _strip_dev(_real_tensor)
    real_init = dist.init_process_group
    dist.init_process_group = lambda backend, device_id=None, **k: real_init('gloo', **k)
    if HANG == 'teardown':
        import threading
        dist.destroy_process_group = lambda *a, **k: threading.Event().wait(3600)


class FakeEngine:
    launch_count, w_dim, z_dim = 0, 8, 8

    def __init__(self, batch):
        self.batch = batch

    def debug_time_gemms(self, reps=10):
        n = 13
        return {'forward': [0.1] * n, 'dgrad': [0.1] * n, 'fir_forward': [0.01] * n, 'fir_backward': [0.01] * n, 'seed': 0.01}


class FakeCore:
    def __init__(self, B, res, C):
        self.engines = [FakeEngine(B)]
        self.B, self.res, self.C = B, res, C
        self.generator_state, self.W, self.X = {}, None, None

    def forward(self, w):
        self.engines[0].launch_count += 64
        return torch.full([self.B, self.C, 4, 4], float(self.engines[0].launch_count // 64)), w      # pixel = number of this call


class FakeAug:
    def __init__(self, c, B):
        self.B, self.res = B, c['img_resolution']
        self.latent_aug = types.SimpleNamespace(module=FakeCore(B, self.res, c['img_channels']))
        self.stats_dataset_w = types.SimpleNamespace(index={f'n{i}': i for i in range(64)})

    def sample_from_inversion(self, paths):
        return torch.zeros([len(paths), 1, 8])

    def set_input(self, data):
        self.data = data

    def forward(self):
        self.latent_aug.module.forward(None)

    def get_output(self):
        return {'A': torch.zeros([self.B, 1, self.res, self.res]), 'B': torch.zeros([self.B, 1, self.res, self.res])}


class FakeBank:
    def __init__(self, Y, index_offset=0):
        self.Y, self.K, self.off = Y, Y.shape[1], index_offset

    def nearest(self, X, k, out=None):
        D = fake_pairwise(X, self.Y).t()
        d, i = torch.topk(D, k, dim=1, largest=False, sorted=True)
        return d, i + self.off


def fake_pairwise(X, Y):
    return ((Y * Y).sum(1)[:, None] + (X * X).sum(1)[None, :]) - 2.0 * (Y @ X.t())


class FakeSearcher:
    graph = None

    def __init__(self, bank, n, k):
        self.bank, self.k = bank, k
        self.world = dist.get_world_size() if dist.is_initialized() else 1

    def __call__(self, X):
        d, i = self.bank.nearest(X, self.k)
        if self.world == 1:
            return d, i
        dl = [torch.empty_like(d) for _ in range(self.world)]
        il = [torch.empty_like(i) for _ in range(self.world)]
        dist.all_gather(dl, d)
        dist.all_gather(il, i)
        dc, ic = torch.cat(dl, 1), torch.cat(il, 1)
        o = torch.sort(dc, dim=1, stable=True).indices[:, :self.k]
        return torch.gather(dc, 1, o), torch.gather(ic, 1, o)

    def close(self):
        pass


def main():
    patch_torch()
    from latentaugment_b200 import engine, parallel
    engine.LatentBank, engine.pairwise_sqdist, parallel.ShardedNearest = FakeBank, fake_pairwise, FakeSearcher
    bench.C5.update(codes=8 * 256, queries=16, dim=8, k=4)
    bench.make_plugin = lambda c, B, local_rank, precision, weights, micro_batches=1: FakeAug(c, min(B, 2))
    bench.time.sleep = lambda s: None
    # the legs size their outputs by the config's batch: keep the fake plugin's batch consistent with it
    for c in bench.CONFIGS.values():
        c['batch'] = 2 * int(os.environ.get('WORLD_SIZE', '1')) if c.get('strong') else 2
        c['img_resolution'] = 8
    if HANG == 'c5' and int(os.environ.get('RANK', '0')) == 0:
        import threading
        bench.c5_leg = lambda *a, **k: threading.Event().wait(3600)
    bench.main()


if __name__ == '__main__':
    main()
