"""Precision and recall of generated-image features against real-image features (DESIGN.md §12).

    python tools/precision_recall.py REAL GEN [--nhood 3]
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/precision_recall.py REAL GEN

REAL and GEN are ``.pt`` (a tensor) or ``.npy`` files of shape [N, K] (detector features, e.g. StyleGAN3's VGG16
embeddings; K a multiple of 64).  Under torchrun every rank reads both files and the work is sharded by rows.
Prints one JSON line (rank 0).
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch
import torch.distributed as dist

from latentaugment_b200.metrics import precision_recall


def load_features(path):
    if path.endswith('.npy'):
        t = torch.from_numpy(np.load(path))
    else:
        t = torch.load(path, map_location='cpu', weights_only=True)
    if not torch.is_tensor(t) or t.dim() != 2:
        raise SystemExit(f'{path}: expected an [N, K] tensor')
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('real')
    ap.add_argument('gen')
    ap.add_argument('--nhood', type=int, default=3)
    a = ap.parse_args()
    rank, world, lr = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(lr)
    dev = torch.device(f'cuda:{lr}')
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    real, gen = load_features(a.real).to(dev), load_features(a.gen).to(dev)
    stats = {}
    p, r = precision_recall(real, gen, a.nhood, stats=stats)
    if rank == 0:
        print(json.dumps({'precision': p, 'recall': r, 'nhood_size': a.nhood, 'n_real': real.shape[0], 'n_gen': gen.shape[0],
                          'dim': real.shape[1], 'n_gpus': world, **stats}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
