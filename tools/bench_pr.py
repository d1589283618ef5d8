"""Benchmark of precision / recall (DESIGN.md §12) against the reference algorithm on the same GPU.

    python tools/bench_pr.py [--n 50000] [--dim 4096] [--nhood 3] [--ref-rows 10000]
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/bench_pr.py ...

Workload: n real + n generated seeded synthetic features of the detector kind (ReLU(0.8 shared + 0.6 noise), rounded to
fp16; correlated, non-negative).  Times each step of both directions with CUDA events after one untimed warm-up of the
whole metric: radii (split candidate pass + exact re-rank) and membership (kEpiMember pass + recheck), each rank on its
shard, the collectives included; reports the slowest rank.  FLOPs are those of the candidate passes computed from the
shapes: 3 bf16 passes x 2 n_rows m K for each step.

Comparator (rank 0 only, not sharded): the reference's compute_pr on the same GPU -- fp16 torch.cdist per row batch of
--ref-rows against column batches of 10 000, each distance block copied to host memory, kthvalue on the CPU for the
radii, ``(dist <= kth).any`` for the membership.  One row batch of each step is timed (host clock around synchronised
work); the full reference time is that times the 4 n / ref_rows row batches of the metric (marked as extrapolated).
With --ref-full the whole reference metric also runs and its P, R are reported.  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch
import torch.distributed as dist

from latentaugment_b200 import metrics, parallel
from latentaugment_b200.engine import FeatureManifold
from oracle import precision_recall as opr


def features(n, K, seed, dev):
    shared = torch.randn([K], generator=torch.Generator().manual_seed(12345))
    out = torch.empty([n, K], dtype=torch.float16)
    g = torch.Generator().manual_seed(seed)
    for b in range(0, n, 8192):
        c = min(8192, n - b)
        out[b:b + c] = torch.relu(0.8 * shared + 0.6 * torch.randn([c, K], generator=g)).half()
    return out.to(dev).float()


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=50000)
    ap.add_argument('--dim', type=int, default=4096)
    ap.add_argument('--nhood', type=int, default=3)
    ap.add_argument('--ref-rows', type=int, default=10000)
    ap.add_argument('--ref-full', action='store_true')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    rank, world, lr = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(lr)
    dev = torch.device(f'cuda:{lr}')
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    real, gen = features(a.n, a.dim, 1, dev), features(a.n, a.dim, 2, dev)

    # untimed warm-up of the whole metric (module load, function attributes, workspaces, communicators)
    stats = {}
    p, r = metrics.precision_recall(real, gen, a.nhood, stats=stats)
    torch.cuda.synchronize()

    def timed(fn):
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return out, ms

    steps = {}
    fallback = {}
    for name, manifold, probes in (('precision', real, gen), ('recall', gen, real)):
        M = FeatureManifold(manifold)
        b, e = parallel.shard_range(M.m, rank, world)

        def radii():
            r2 = M.radii(b, e, a.nhood)
            if world > 1:
                per = -(-M.m // world)
                piece = torch.zeros([per], device=dev)
                piece[:e - b] = r2
                pieces = [torch.empty_like(piece) for _ in range(world)]
                dist.all_gather(pieces, piece)
                r2 = torch.cat([pieces[k][:parallel.shard_range(M.m, k, world)[1] - parallel.shard_range(M.m, k, world)[0]]
                                for k in range(world)])
            return r2
        r2, ms_r = timed(radii)
        fb_r = int(M.fallback.item())
        pb, pe = parallel.shard_range(probes.shape[0], rank, world)
        _, ms_m = timed(lambda: M.member(probes[pb:pe], r2))
        fb_m = int(M.fallback.item()) - fb_r
        if world > 1:
            t = torch.tensor([fb_r, fb_m], device=dev, dtype=torch.int64)
            dist.all_reduce(t)
            fb_r, fb_m = t.tolist()
        steps[name] = {'radii_ms': ms_r, 'member_ms': ms_m}
        fallback[name] = {'radii': fb_r, 'member': fb_m}
        del M
    total_ms = sum(s['radii_ms'] + s['member_ms'] for s in steps.values())
    step_flops = 3 * 2.0 * a.n * a.n * a.dim                          # one step of one direction (all ranks)

    res = None
    if rank == 0:
        res = {'metric': 'precision_recall', 'n_gpus': world, 'n_real': a.n, 'n_gen': a.n, 'dim': a.dim, 'nhood': a.nhood,
               'card': card(), 'precision': p, 'recall': r, 'steps_ms': steps, 'fallback': fallback, 'metric_ms': total_ms,
               'candidate_pass_flops_per_step': step_flops,
               'candidate_pass_tflops': 4 * step_flops / (total_ms * 1e-3) / 1e12}
        # reference comparator: one row batch of each step on this GPU, host copies and CPU kthvalue included
        rows = min(a.ref_rows, a.n)
        r16, g16 = real.half(), gen.half()
        opr.compute_distances(r16[:256], r16[:20000], 10000).float().kthvalue(a.nhood + 1)     # warm-up (kernels, allocator)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dist_b = opr.compute_distances(r16[:rows], r16, 10000)
        kth = dist_b.to(torch.float32).kthvalue(a.nhood + 1).values.to(torch.float16)
        t_radii = time.perf_counter() - t0
        kth_all = torch.full([a.n], 65504.0, dtype=torch.float16)
        kth_all[:rows] = kth
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dist_b = opr.compute_distances(g16[:rows], r16, 10000)
        (dist_b <= kth_all).any(dim=1)
        t_member = time.perf_counter() - t0
        batches = -(-a.n // rows)
        res['reference'] = {'method': f'fp16 torch.cdist, row batch {rows} x column batches of 10000, host copies, CPU kthvalue',
                            'radii_batch_s': t_radii, 'member_batch_s': t_member, 'row_batches_per_step': batches,
                            'metric_s_extrapolated': 2 * batches * (t_radii + t_member)}
        res['speedup_vs_reference_extrapolated'] = res['reference']['metric_s_extrapolated'] / (total_ms * 1e-3)
        if a.ref_full:
            t0 = time.perf_counter()
            ref = opr.compute_pr_reference(real, gen, a.nhood, row_batch_size=rows, device=dev)
            res['reference'].update(precision=ref['precision'], recall=ref['recall'], metric_s_measured=time.perf_counter() - t0)
        print(json.dumps(res))
        if a.out:
            os.makedirs(os.path.dirname(a.out) or '.', exist_ok=True)
            with open(a.out, 'w') as f:
                json.dump(res, f, indent=1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
