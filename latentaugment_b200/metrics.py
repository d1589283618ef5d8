"""Precision and recall of generated images (Kynkäänniemi et al. 2019, StyleGAN3's ``compute_pr``) on detector features.

``precision_recall`` computes, exactly and deterministically, the metric of DESIGN.md §12: the features are rounded to
fp16 as the reference rounds them; a manifold point's radius is its (nhood+1)-th smallest squared distance over the
manifold (itself included); a probe counts when some manifold ball holds it under the reference's comparison of fp16
distances.  Precision uses the real features as the manifold and the generated ones as probes; recall the reverse.
"""
import torch
import torch.distributed as dist

from .parallel import shard_range


def _manifold(Y):
    from .engine import FeatureManifold
    return FeatureManifold(Y)


def _direction(manifold, probes, nhood_size, rank, world, group):
    """(members among this rank's probe shard, fallback count) of one direction.  Manifold rows are sharded for the
    radii; one all_gather makes the radii whole on every rank."""
    M = _manifold(manifold)
    b, e = shard_range(M.m, rank, world)
    r2 = M.radii(b, e, nhood_size)
    if world > 1:
        per = -(-M.m // world)                          # equal-sized pieces for the collective
        piece = torch.zeros([per], device=r2.device)
        piece[:e - b] = r2
        pieces = [torch.empty_like(piece) for _ in range(world)]
        dist.all_gather(pieces, piece, group=group)
        r2 = torch.cat([pieces[k][:shard_range(M.m, k, world)[1] - shard_range(M.m, k, world)[0]] for k in range(world)])
    pb, pe = shard_range(probes.shape[0], rank, world)
    members = M.member(probes[pb:pe], r2).sum(dtype=torch.int64)
    return members, M.fallback.to(torch.int64).sum()


def precision_recall(real_features, gen_features, nhood_size=3, group=None, stats=None):
    """(precision, recall) of ``gen_features`` against ``real_features`` ([N, K] tensors on the GPU, K a multiple of 64).

    With an initialised process group every rank passes the same features; each computes the radii of its shard of
    manifold rows and the membership of its shard of probes (``parallel.shard_range``), the radii are all-gathered and
    the member counts all-reduced, and every rank returns the same result.  ``stats``: a dict that receives the number
    of queries scanned exhaustively (``fallback_precision`` / ``fallback_recall``, summed over ranks)."""
    assert real_features.dim() == 2 and gen_features.dim() == 2 and real_features.shape[1] == gen_features.shape[1]
    distributed = group is not None or (dist.is_available() and dist.is_initialized())
    world = dist.get_world_size(group) if distributed else 1
    rank = dist.get_rank(group) if distributed else 0
    p, fp = _direction(real_features, gen_features, nhood_size, rank, world, group)
    r, fr = _direction(gen_features, real_features, nhood_size, rank, world, group)
    counts = torch.stack([p, r, fp, fr])
    if world > 1:
        dist.all_reduce(counts, group=group)
    counts = counts.tolist()
    if stats is not None:
        stats.update(fallback_precision=counts[2], fallback_recall=counts[3])
    return counts[0] / gen_features.shape[0], counts[1] / real_features.shape[0]
