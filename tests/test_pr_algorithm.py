"""CPU restatement of the two GPU steps of the precision / recall metric (csrc/distance.cu, DESIGN.md §12), checked
against the exhaustive fp64 definition (oracle/precision_recall.py) on adversarial and correlated feature sets.

* Candidate scores on split planes: s^ = |y|^2 - 2 (<xh,yh> + <xl,yh> + <xh,yl>) with fp32 accumulation, and the margin
  eps = split_eps_coef(K) |x| max|y| + 6e-7 (|x|^2 + max|y|^2) the kernels use.
* Membership (kEpiMember + member_recheck_kernel): a definite hit when s^ - (T_j - |x|^2) <= -(eps + 2.4e-7 T_j), ambiguous
  columns listed per probe (kMemberCap), overflowed probes rescanned, the rest rechecked with the exact distance.
* Radii (kEpiTopK + rerank_kernel with the split eps): two candidates per 32-point chunk, cut = 8th smallest + 2 eps,
  overflowed chunks and the survivors re-ranked exactly (kMaxList / kMaxOvf bound the lists).
"""
import math

import pytest
import torch

from oracle import precision_recall as opr

K_MEMBER_CAP, K_MAX_LIST, K_MAX_OVF = 256, 512, 128


def split_eps_coef(K):
    return 3.0518e-5 + K * 3.612e-7


def planes(X):
    hi = X.float().to(torch.bfloat16).float()
    lo = (X.float() - hi).to(torch.bfloat16).float()
    return hi, lo


def split_scores(X, Y):
    """s^ [n, m] fp32 and the per-row eps (X, Y fp16-valued)."""
    xh, xl = planes(X)
    yh, yl = planes(Y)
    acc = xh @ yh.T + xl @ yh.T + xh @ yl.T                      # fp32 accumulation
    yy = (Y.double() ** 2).sum(1).float()
    xx = (X.double() ** 2).sum(1).float()
    ymax = yy.max()
    s = yy[None, :] - 2.0 * acc
    eps = split_eps_coef(X.shape[1]) * xx.sqrt() * ymax.sqrt() + 6e-7 * (xx + ymax)
    return s, xx, eps


def member_algorithm(X, Y, r2, eps_scale=1.0, cap=K_MEMBER_CAP, T=None):
    """(member [n] bool, probes rescanned exhaustively).  ``T`` overrides the thresholds of r2 (tests of the decision
    step alone)."""
    s, xx, eps = split_scores(X, Y)
    T = opr.threshold(r2) if T is None else T
    mgc = torch.where(torch.isinf(T), torch.zeros_like(T), 2.4e-7 * T)
    d = s - (T[None, :] - xx[:, None])
    mg = eps_scale * (eps[:, None] + mgc[None, :])
    hit = (d <= -mg).any(1)
    amb = d <= mg
    exact = opr.definition_sqdist(X, Y) <= T[None, :]
    member = hit.clone()
    fallback = 0
    for i in torch.nonzero(~hit).flatten().tolist():
        cols = torch.nonzero(amb[i]).flatten()
        if cols.numel() > cap:
            fallback += 1
            member[i] = exact[i].any()
        else:
            member[i] = exact[i, cols].any()
    return member, fallback


def radii_algorithm(Y, nhood):
    """(r2 [m], survivors per query, queries scanned exhaustively) of the candidate pass + exact re-rank."""
    m = Y.shape[0]
    k = nhood + 1
    s, xx, eps = split_scores(Y, Y)
    exact = opr.definition_sqdist(Y, Y)
    pad = (-m) % 32
    sp = torch.nn.functional.pad(s, [0, pad], value=float('inf')).view(m, -1, 32)
    top2, _ = sp.topk(2, dim=2, largest=False)                   # ascending per chunk
    pairs = top2.reshape(m, -1)
    thr = pairs.kthvalue(8, dim=1).values if pairs.shape[1] >= 8 else torch.full([m], float('inf'))
    cut = thr + 2 * eps
    ovf = top2[:, :, 1] <= cut[:, None]                          # the chunk may hide more: rescanned
    r2 = torch.empty(m)
    survivors, fallback = [], 0
    chunk_of = torch.arange(m) // 32
    for i in range(m):
        keep = (s[i] <= cut[i]) & ~ovf[i, chunk_of]
        top2_cols = torch.zeros(m, dtype=torch.bool)            # only the two listed candidates of a chunk can survive
        cols = sp[i].topk(2, dim=1, largest=False).indices + torch.arange(sp.shape[1])[:, None] * 32
        top2_cols[cols.flatten()[cols.flatten() < m]] = True
        keep &= top2_cols
        n_ovf = int(ovf[i].sum())
        survivors.append(int(keep.sum()))
        if math.isinf(thr[i]) or n_ovf > K_MAX_OVF or int(keep.sum()) > K_MAX_LIST:
            fallback += 1
            cand = torch.ones(m, dtype=torch.bool)
        else:
            cand = keep | ovf[i, chunk_of]
        vals = exact[i][cand]
        r2[i] = vals.sort().values[k - 1]
    return r2, survivors, fallback


def correlated(n, K, seed, shared=None):
    """Non-negative, highly correlated detector-like features: ReLU(0.8 shared + 0.6 noise), rounded to fp16."""
    g = torch.Generator().manual_seed(seed)
    if shared is None:
        shared = torch.randn([K], generator=torch.Generator().manual_seed(12345))
    return torch.relu(0.8 * shared + 0.6 * torch.randn([n, K], generator=g)).to(torch.float16).float()


def fp16_vector_with_sqnorm(target, K):
    """An fp16-valued [K] vector whose squared norm is exactly ``target`` (a multiple of 0.25), greedily from the top."""
    v, rem, t = torch.zeros(K, dtype=torch.float64), float(target), 0
    while rem > 0:
        h = torch.tensor(math.sqrt(rem)).to(torch.float16)
        while float(h) ** 2 > rem:                               # step down one fp16 value at a time
            h = (h.view(torch.int16) - 1).view(torch.float16)
        c = float(h)
        c = math.floor(c * 2) / 2 if c < 2048 else c
        assert c > 0 and t < K
        v[t] = c
        rem -= c * c
        t += 1
    assert (v * v).sum().item() == target
    return v.float()


def boundary_cases(K):
    """(manifold [2, K], r2 [2], probes [p, K], expected [p]): manifold point 0 at the origin with h(r2) = H, probes at
    squared distance exactly b^2, one fp32 step inside and outside; point 1 far away with radius 0."""
    cases = []
    far = torch.zeros(K)
    far[K - 1] = 60000.0
    for H, b, even in ((2048.0, 2049.0, True), (2050.0, 2051.0, False), (0.5, 0.50048828125, True),
                       (65504.0, 65520.0, False)):
        b2 = b * b
        ulp = float(torch.nextafter(torch.tensor(b2, dtype=torch.float32), torch.tensor(float('inf'))) - b2)
        for d2, exp in ((b2, even), (b2 - ulp, True), (b2 + ulp, False)):
            if d2 * 4 != math.floor(d2 * 4):
                continue                                     # not reachable by fp16 squares at this scale
            probe = fp16_vector_with_sqnorm(d2, K)
            cases.append((torch.stack([torch.zeros(K), far]), torch.tensor([H * H, 0.0]), probe[None], [exp]))
    # beyond the fp16 range: h(r2) = inf admits every distance, h(r2) = 65504 none beyond 65520
    probe = fp16_vector_with_sqnorm(65504.0 ** 2 + 1447.0 ** 2, K)
    cases.append((torch.stack([torch.zeros(K), far]), torch.tensor([65600.0 ** 2, 0.0]), probe[None], [True]))
    return cases


@pytest.mark.parametrize('K', [64, 512, 4096])
def test_membership_boundaries_exact(K):
    for Y, r2, P, expected in boundary_cases(K):
        ref = opr.definition_member(P, Y, r2)
        got, _ = member_algorithm(P, Y, r2)
        assert ref.tolist() == expected, (r2, (P.double() ** 2).sum(1))
        assert got.tolist() == expected


def test_threshold_rule_matches_h():
    """d2 <= T_j  <=>  h(d2) <= h(r2_j) on every fp32 value around the edges of many radii."""
    g = torch.Generator().manual_seed(3)
    r2 = torch.cat([torch.rand(200, generator=g) * 10.0 ** torch.randint(-8, 10, [200], generator=g),
                    torch.tensor([0.0, 65504.0 ** 2, 65520.0 ** 2, 65519.0 ** 2, 2.0 ** -50])])
    T = opr.threshold(r2)
    for j in range(r2.numel()):
        H = opr.h(r2[j:j + 1])
        if torch.isinf(T[j]):
            assert torch.isinf(H).all()
            continue
        d = T[j].repeat(5)
        d = torch.stack([torch.nextafter(d[0], torch.tensor(0.0)), d[0], torch.nextafter(d[0], torch.tensor(float('inf')))])
        assert (opr.h(d) <= H).tolist() == [True, True, False], (r2[j], T[j])


@pytest.mark.parametrize('K,n,m', [(64, 37, 45), (512, 129, 300), (4096, 61, 200)])
def test_membership_and_radii_match_definition(K, n, m):
    shared = torch.randn([K], generator=torch.Generator().manual_seed(K))
    Y = correlated(m, K, 1, shared)
    Y[5] = Y[6] = Y[7] = Y[8]                                   # duplicates: radius 0 at nhood 3
    X = torch.cat([correlated(n - 2, K, 2, shared), Y[5:6], Y[20:21]])   # probes on manifold points
    for nhood in (1, 3, 7):
        r2, surv, fb = radii_algorithm(Y, nhood)
        ref = opr.definition_radii(Y, nhood)
        assert torch.equal(r2, ref)
        assert fb == 0 or m < 8 * 32 // 2          # fewer than 8 candidates: every query scans the (small) manifold
        if nhood == 3:
            assert r2[5] == 0.0
        got, _ = member_algorithm(X, Y, ref)
        assert torch.equal(got, opr.definition_member(X, Y, ref))
        assert got[-2] and got[-1]


def test_distances_beyond_fp16_range():
    """Features near the top of the fp16 range: distances above 65520 saturate h to +inf on both sides."""
    K = 64
    g = torch.Generator().manual_seed(5)
    Y = (torch.rand([40, K], generator=g) * 30000).to(torch.float16).float()
    X = (torch.rand([33, K], generator=g) * 30000).to(torch.float16).float()
    r2 = opr.definition_radii(Y, 3)
    assert (opr.h(r2) == float('inf')).all()                    # every radius beyond fp16: every probe is a member
    got, _ = member_algorithm(X, Y, r2)
    assert got.all() and torch.equal(got, opr.definition_member(X, Y, r2))
    r2 = torch.full([40], 65504.0 ** 2)                         # h = 65504: only distances below 65520 count
    got, _ = member_algorithm(X, Y, r2)
    assert torch.equal(got, opr.definition_member(X, Y, r2)) and not got.all()


def test_zero_margin_gets_decisions_wrong():
    """Without the margin the approximate scores decide pairs at a threshold edge wrongly: the margin is needed.  Every
    point's threshold is set to the exact distance of one probe, so that probe sits exactly on the edge."""
    K, m, n = 4096, 256, 400
    shared = torch.randn([K], generator=torch.Generator().manual_seed(7))
    Y = correlated(m, K, 1, shared)
    X = correlated(n, K, 2, shared)
    d2 = opr.definition_sqdist(X, Y)
    T = d2.min(0).values
    ref = (d2 <= T[None, :]).any(1)
    right, _ = member_algorithm(X, Y, None, T=T)
    wrong, _ = member_algorithm(X, Y, None, eps_scale=0.0, T=T)
    assert torch.equal(right, ref)
    assert not torch.equal(wrong, ref)


def test_correlated_features_never_fall_back():
    """On the correlated detector-like features at m = 8 192 no query exceeds kMaxList / kMaxOvf in the radii and no
    probe overflows its ambiguous list: the fallback count is 0 (a subset of queries, all m points as the manifold)."""
    K, m = 4096, 8192
    Y = correlated(m, K, 11)
    q = torch.arange(0, m, 97)                                 # 85 manifold rows as radii queries
    s, xx, eps = split_scores(Y[q], Y)
    pad = (-m) % 32
    top2 = torch.nn.functional.pad(s, [0, pad], value=float('inf')).view(q.numel(), -1, 32).topk(2, dim=2, largest=False).values
    thr = top2.reshape(q.numel(), -1).kthvalue(8, dim=1).values
    cut = thr + 2 * eps
    novf = (top2[:, :, 1] <= cut[:, None]).sum(1)
    surv = ((top2[:, :, 0] <= cut[:, None]) & (top2[:, :, 1] > cut[:, None])).sum(1)
    assert int(novf.max()) <= K_MAX_OVF and int(surv.max()) <= K_MAX_LIST, (novf.max(), surv.max())
    # membership of fresh probes against all m balls (radii from fp32 distances: they only place the thresholds)
    Yh = Y.to(torch.float16).float()
    yy = (Yh * Yh).sum(1)
    r2 = torch.cat([(yy[None, :] + yy[b:b + 1024, None] - 2 * Yh[b:b + 1024] @ Yh.T).kthvalue(4, dim=1).values
                    for b in range(0, m, 1024)])
    X = correlated(300, K, 12)
    sX, xxX, epsX = split_scores(X, Y)
    T = opr.threshold(r2)
    d = sX - (T[None, :] - xxX[:, None])
    mg = epsX[:, None] + 2.4e-7 * T[None, :]
    undecided = ~(d <= -mg).any(1)
    amb = (d.abs() <= mg).sum(1)
    assert (int(amb[undecided].max()) if undecided.any() else 0) <= K_MEMBER_CAP
    print(f'radii survivors median {int(surv.median())} max {int(surv.max())}, overflowed chunks max {int(novf.max())}; '
          f'probes undecided after the pass {int(undecided.sum())} of 300, ambiguous per undecided probe max '
          f'{int(amb[undecided].max()) if undecided.any() else 0}')
