"""Precision / recall on the GPU (csrc/distance.cu, DESIGN.md §12): radii and membership flags bit-identical to the
exhaustive fp64 definition (oracle/precision_recall.py), the adversarial sets of tests/test_pr_algorithm.py through the
kernels, the metric against the definition and the literal reference run on the same GPU, and the fallback count on
correlated detector-like features."""
import pytest
import torch

from oracle import precision_recall as opr
from test_pr_algorithm import boundary_cases, correlated

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _manifold(Y):
    from latentaugment_b200.engine import FeatureManifold
    return FeatureManifold(Y.to(DEV))


@pytest.mark.parametrize('K', [512, 2048, 4096])
@pytest.mark.parametrize('n,m', [(333, 517), (97, 200)])
def test_radii_and_membership_bit_identical(K, n, m):
    shared = torch.randn([K], generator=torch.Generator().manual_seed(K + m))
    Y = correlated(m, K, 1, shared)
    Y[10] = Y[11] = Y[12] = Y[13]                                  # duplicates: radius 0 up to nhood 3
    X = torch.cat([correlated(n - 2, K, 2, shared), Y[10:11], Y[50:51]])
    M = _manifold(Y)
    Yd = opr.as_definition_input(Y)
    for nhood in (1, 3, 7):
        r2 = M.radii(0, m, nhood).cpu()
        ref = opr.definition_radii(Yd, nhood)
        assert torch.equal(r2, ref), (nhood, (r2 != ref).sum().item())
        part = M.radii(m // 3, m // 3 + 41, nhood).cpu()          # a shard of rows gives the same radii
        assert torch.equal(part, ref[m // 3:m // 3 + 41])
        mem = M.member(X.to(DEV), r2.to(DEV)).cpu().bool()
        assert torch.equal(mem, opr.definition_member(opr.as_definition_input(X), Yd, ref)), nhood
        assert mem[-2] and mem[-1]


@pytest.mark.parametrize('K', [512, 4096])
def test_adversarial_boundaries_through_the_kernels(K):
    for Y, r2, P, expected in boundary_cases(K):
        M = _manifold(Y)
        got = M.member(P.to(DEV), r2.to(DEV)).cpu().bool().tolist()
        assert got == expected, (r2, (P.double() ** 2).sum(1))


def test_metric_equals_definition_and_reference_within_band():
    from latentaugment_b200.metrics import precision_recall
    K = 2048
    shared = torch.randn([K], generator=torch.Generator().manual_seed(9))
    real, gen = correlated(3000, K, 21, shared), correlated(2500, K, 22, shared)
    stats = {}
    p, r = precision_recall(real.to(DEV), gen.to(DEV), 3, stats=stats)
    p0, r0 = opr.definition_pr(real, gen, 3)
    assert (p, r) == (p0, r0)
    ref = opr.compute_pr_reference(real, gen, 3, device=DEV)       # fp16 cdist on the GPU, host kthvalue
    for name, manifold, probes, val in (('precision', real, gen, p), ('recall', gen, real, r)):
        band = opr.rounding_band(probes, manifold, 3)
        mine = opr.definition_member(opr.as_definition_input(probes), opr.as_definition_input(manifold),
                                     opr.definition_radii(opr.as_definition_input(manifold), 3))
        differ = mine != ref[name + '_pred']
        assert not (differ & ~band).any(), (name, int((differ & ~band).sum()))
        assert abs(val - ref[name]) <= band.sum().item() / probes.shape[0] + 1e-12
    assert stats == {'fallback_precision': 0, 'fallback_recall': 0}


def test_no_fallback_on_correlated_features_at_8192():
    K, m = 4096, 8192
    Y = correlated(m, K, 31)
    X = correlated(2000, K, 32)
    M = _manifold(Y)
    r2 = M.radii(0, m, 3)
    M.member(X.to(DEV), r2)
    torch.cuda.synchronize()
    assert int(M.fallback.item()) == 0
    sel = torch.arange(0, m, 61)
    Yd = opr.as_definition_input(Y)
    assert torch.equal(r2.cpu()[sel], opr.definition_sqdist(Yd[sel], Yd).kthvalue(4, dim=1).values)
