"""Host-side checks of the precision / recall feature: the C-ABI planners and argument rejections (no device needed),
the definition against the literal reference restatement, and the sharded ``metrics.precision_recall`` under a 2-rank
gloo group with the CUDA calls replaced by the CPU definition."""
import ctypes
import os

import torch

from oracle import precision_recall as opr


def test_pr_planners_and_rejections_on_the_host():
    from latentaugment_b200 import _lib
    lib = _lib.load()
    n = ctypes.c_size_t(0)
    assert lib.la_pr_radii_workspace_bytes(8192, 50000, 4096, 3, ctypes.byref(n)) == 0
    cand = 8192 * ((50000 + 255) // 256 * 16) * 8                      # two candidates per 32 points, score + index
    planes = 8192 * 4096 * 2 * 2                                       # query hi + lo
    assert cand + planes <= n.value < cand + planes + 8 * 2 ** 20
    radii = n.value
    assert lib.la_pr_member_workspace_bytes(8192, 50000, 4096, ctypes.byref(n)) == 0
    assert planes + 8192 * 256 * 4 <= n.value < radii                 # bounded per-probe lists, no candidate lists
    assert lib.la_pr_member_workspace_bytes(8192, 50000, 4000, ctypes.byref(n)) != 0          # K % 64
    for nhood, m, K in ((0, 100, 512), (8, 100, 512), (3, 3, 512), (7, 7, 512), (3, 100, 96)):
        assert lib.la_pr_radii_workspace_bytes(16, m, K, nhood, ctypes.byref(n)) != 0, (nhood, m, K)
        assert lib.la_last_error()
    assert lib.la_pr_radii_workspace_bytes(16, 4, 512, 3, ctypes.byref(n)) == 0              # m = nhood + 1 is enough
    # the entries reject the same shapes and a misaligned workspace before touching the device
    buf = ctypes.create_string_buffer(4096)
    p = ctypes.c_void_p(ctypes.addressof(buf))
    odd = ctypes.c_void_p(ctypes.addressof(buf) + 8 if ctypes.addressof(buf) % 1024 == 0 else ctypes.addressof(buf))
    assert lib.la_pr_radii(p, 16, p, p, p, 3, 512, 3, p, 1 << 40, p, None, None) != 0          # m < nhood + 1
    assert lib.la_pr_radii(p, 16, p, p, p, 100, 512, 3, odd, 1 << 40, p, None, None) != 0      # alignment
    assert lib.la_pr_member(p, 16, p, p, p, p, 100, 100, p, 1 << 40, p, None, None) != 0       # K % 64
    assert lib.la_pr_member(p, 16, p, p, p, p, 100, 512, odd, 1 << 40, p, None, None) != 0     # alignment
    assert lib.la_pr_member(p, 16, p, p, p, p, 100, 512, p, 1024, p, None, None) != 0          # workspace size


def _features(n, K, seed, shared):
    g = torch.Generator().manual_seed(seed)
    return torch.relu(0.8 * shared + 0.6 * torch.randn([n, K], generator=g))


def test_definition_matches_reference_outside_the_rounding_band():
    """The literal compute_pr restatement (fp16 cdist on the CPU) and the definition agree on every probe outside the
    counted rounding band, and |dP|, |dR| <= band / n."""
    K = 512
    shared = torch.randn([K], generator=torch.Generator().manual_seed(1))
    real, gen = _features(700, K, 2, shared), _features(650, K, 3, shared)
    ref = opr.compute_pr_reference(real, gen, 3, row_batch_size=256, col_batch_size=300)
    p, r = opr.definition_pr(real, gen, 3)
    for name, manifold, probes, val in (('precision', real, gen, p), ('recall', gen, real, r)):
        band = opr.rounding_band(probes, manifold, 3)
        mine = opr.definition_member(opr.as_definition_input(probes), opr.as_definition_input(manifold),
                                     opr.definition_radii(opr.as_definition_input(manifold), 3))
        differ = mine != ref[name + '_pred']
        assert not (differ & ~band).any(), name
        assert abs(val - ref[name]) <= band.sum().item() / probes.shape[0] + 1e-12
        assert 0.05 < val < 0.95                                        # the data exercises both outcomes


class _CpuManifold:
    """FeatureManifold stand-in: the exhaustive definition on the CPU, recording which rows each rank asked for."""
    calls = []

    def __init__(self, Y):
        self.Y = opr.as_definition_input(Y)
        self.m = Y.shape[0]
        self.fallback = torch.zeros([1], dtype=torch.int32)

    def radii(self, begin, end, nhood_size):
        _CpuManifold.calls.append(('radii', begin, end))
        return opr.definition_sqdist(self.Y[begin:end], self.Y).kthvalue(nhood_size + 1, dim=1).values

    def member(self, X, r2):
        _CpuManifold.calls.append(('member', X.shape[0]))
        return opr.definition_member(opr.as_definition_input(X), self.Y, r2).to(torch.uint8)


def _pr_worker(rank, world, port, q):
    import torch.distributed as dist

    from latentaugment_b200 import metrics, parallel
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    metrics._manifold = _CpuManifold
    gathers, reduces = [], []
    ag, ar = dist.all_gather, dist.all_reduce
    dist.all_gather = lambda *a, **k: (gathers.append(1), ag(*a, **k))[1]
    dist.all_reduce = lambda *a, **k: (reduces.append(1), ar(*a, **k))[1]
    K = 64
    shared = torch.randn([K], generator=torch.Generator().manual_seed(4))
    real, gen = _features(101, K, 5, shared), _features(77, K, 6, shared)
    stats = {}
    p, r = metrics.precision_recall(real, gen, 3, stats=stats)
    p0, r0 = opr.definition_pr(real, gen, 3)
    expect = [('radii',) + parallel.shard_range(101, rank, world), ('member', parallel.shard_range(77, rank, world)[1] - parallel.shard_range(77, rank, world)[0]),
              ('radii',) + parallel.shard_range(77, rank, world), ('member', parallel.shard_range(101, rank, world)[1] - parallel.shard_range(101, rank, world)[0])]
    ok = (p == p0 and r == r0 and _CpuManifold.calls == expect and len(gathers) == 2 and len(reduces) == 1
          and stats == {'fallback_precision': 0, 'fallback_recall': 0})
    q.put((rank, bool(ok), (p, r, p0, r0, _CpuManifold.calls, len(gathers), len(reduces))))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_precision_recall_gloo_world2():
    """Each rank computes the radii of its manifold rows and the membership of its probes (parallel.shard_range); one
    all_gather of the radii per direction and ONE all_reduce of the counts give every rank the single-process result."""
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_pr_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert [(r, ok) for r, ok, _ in res] == [(0, True), (1, True)], res
