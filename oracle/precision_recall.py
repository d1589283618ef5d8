"""Oracle restatement of the precision / recall metric.  TEST INFRASTRUCTURE (see oracle/__init__.py).

Two functions:

* ``compute_pr_reference`` restates StyleGAN3's ``metrics/precision_recall.py::compute_pr`` (with its
  ``compute_distances``; public NVlabs/stylegan3 code, which the LatentAugment tree copies into
  ``metrics/precision_recall.py:19-85``).  It was restated from the public code, not run from the reference tree, and
  keeps the single-process path: features cast with ``.to(torch.float16)``, ``torch.cdist`` on fp16 row batches against
  fp16 column batches, each distance block copied to host memory, ``kthvalue(nhood_size + 1)`` in fp32 on the host
  rounded back to fp16, and ``(dist <= kth).any(dim=1)`` on fp16 distances.
* ``definition_*`` compute the metric this package defines (DESIGN.md §12) exhaustively in fp64 on the CPU: distances
  ``(|y|^2 + |x|^2) - 2 <x,y>`` with each sum in fp64 rounded once to fp32, radii as the (nhood+1)-th smallest distance,
  and membership ``h(d2) <= h(r2)`` with ``h(v) = fp16(sqrt(max(v, 0)))``.

``rounding_band`` counts the probes whose reference decision may legitimately differ from the definition.
"""
import torch


def compute_distances(row_features, col_features, col_batch_size):
    """``compute_distances`` of the reference with num_gpus = 1, rank = 0 (host copies included)."""
    num_cols = col_features.shape[0]
    num_batches = (num_cols - 1) // col_batch_size + 1
    col_batches = torch.nn.functional.pad(col_features, [0, 0, 0, -num_cols % num_batches]).chunk(num_batches)
    dist_batches = []
    for col_batch in col_batches:
        dist_batch = torch.cdist(row_features.unsqueeze(0), col_batch.unsqueeze(0))[0]
        dist_batches.append(dist_batch.cpu())
    return torch.cat(dist_batches, dim=1)[:, :num_cols]


def compute_pr_reference(real_features, gen_features, nhood_size=3, row_batch_size=10000, col_batch_size=10000, device=None):
    """{'precision', 'recall', 'precision_pred', 'recall_pred'} by the reference algorithm (the per-probe decisions
    included)."""
    device = device or real_features.device
    real_features = real_features.to(torch.float16).to(device)
    gen_features = gen_features.to(torch.float16).to(device)
    results = {}
    for name, manifold, probes in [('precision', real_features, gen_features), ('recall', gen_features, real_features)]:
        kth = []
        for manifold_batch in manifold.split(row_batch_size):
            dist = compute_distances(manifold_batch, manifold, col_batch_size)
            kth.append(dist.to(torch.float32).kthvalue(nhood_size + 1).values.to(torch.float16))
        kth = torch.cat(kth)
        pred = []
        for probes_batch in probes.split(row_batch_size):
            dist = compute_distances(probes_batch, manifold, col_batch_size)
            pred.append((dist <= kth).any(dim=1))
        results[name] = float(torch.cat(pred).to(torch.float32).mean())
        results[name + '_pred'] = torch.cat(pred)
    return results


def as_definition_input(features):
    """The caller's features rounded to fp16 as the reference rounds them, held as fp64 (exact)."""
    return features.to(torch.float16).to(torch.float64)


def definition_sqdist(X, Y):
    """[n, m] fp32 ``(|y|^2 + |x|^2) - 2 <x,y>`` with each sum in fp64 rounded once to fp32 (X, Y fp16-valued)."""
    X, Y = X.double(), Y.double()
    xx = (X * X).sum(1).float()
    yy = (Y * Y).sum(1).float()
    dot = (X @ Y.T).float()
    return (yy[None, :] + xx[:, None]) - 2.0 * dot


def definition_radii(Y, nhood_size=3):
    """r2_j = the (nhood+1)-th smallest distance of manifold point j over the whole manifold (itself included)."""
    return definition_sqdist(Y, Y).kthvalue(nhood_size + 1, dim=1).values


def _f16(bits):
    return bits.to(torch.int16).view(torch.float16).double()


def h(v):
    """fp16(sqrt(max(v, 0))), round to nearest even, saturating to +inf.  The fp64 root of an fp32 value never lands on
    an fp16 midpoint unless the exact root does, so one correct rounding of it is exact; torch's fp64 -> fp16 conversion
    goes through fp32 (two roundings), hence the explicit rounding against the midpoint."""
    s = torch.sqrt(v.double().clamp_min(0))
    bits = s.to(torch.float16).view(torch.int16).to(torch.int32)       # within one fp16 step of the answer
    lo_bits = torch.where(_f16(bits) > s, bits - 1, bits)
    lo = _f16(lo_bits)
    hi = torch.where(lo_bits == 0x7bff, torch.full_like(lo, 65536.0), _f16(lo_bits + 1))
    mid = 0.5 * (lo + hi)
    up = (s > mid) | ((s == mid) & (lo_bits % 2 == 1))
    return _f16(torch.where(up, lo_bits + 1, lo_bits)).to(torch.float16)


def threshold(r2):
    """T_j: h(d2) <= h(r2_j) exactly when d2 <= T_j (fp32 d2).  b = upper edge of the fp16 rounding interval of h(r2_j);
    T_j = b^2 (exact in fp32) when h(r2_j) has an even significand, else the fp32 value just below b^2; +inf for h = inf."""
    H = h(r2)
    bits = H.view(torch.int16).to(torch.int32)
    nxt = (bits + 1).to(torch.int16).view(torch.float16).double()
    nxt = torch.where(bits == 0x7bff, torch.full_like(nxt, 65536.0), nxt)
    b = 0.5 * (H.double() + nxt)
    T = (b * b).float()
    T = torch.where((bits & 1) == 1, torch.nextafter(T, torch.zeros_like(T)), T)
    return torch.where(torch.isinf(H), torch.full_like(T, float('inf')), T)


def definition_member(X, Y, r2):
    """[n] bool: probe i is in some manifold ball, h(d2(x_i, y_j)) <= h(r2_j)."""
    return (definition_sqdist(X, Y) <= threshold(r2)[None, :]).any(1)


def definition_pr(real, gen, nhood_size=3):
    real, gen = as_definition_input(real), as_definition_input(gen)
    p = definition_member(gen, real, definition_radii(real, nhood_size)).double().mean().item()
    r = definition_member(real, gen, definition_radii(gen, nhood_size)).double().mean().item()
    return p, r


def rounding_band(X, Y, nhood_size=3, tau=2.0 ** -8):
    """[n] bool: probes whose decision changes when every distance may move by the relative amount ``tau`` (the fp16
    arithmetic of the reference's cdist: a few fp16 ulps).  Order statistics move by at most the same relative amount,
    so outside this band the reference and the definition agree."""
    X, Y = as_definition_input(X), as_definition_input(Y)
    d = definition_sqdist(X, Y).double().clamp_min(0).sqrt()
    r = definition_radii(Y, nhood_size).double().clamp_min(0).sqrt()
    sure_in = (d * (1 + tau) < r[None, :] * (1 - tau)).any(1)
    sure_out = (d * (1 - tau) > r[None, :] * (1 + tau)).all(1)
    return ~(sure_in | sure_out)
