"""Precision and recall of generated-image features against real-image features (DESIGN.md §12).

    python tools/precision_recall.py REAL GEN [--nhood 3]
    python tools/precision_recall.py --images REAL GEN --vgg_state vgg16.pth [--precision bf16] [--split train --modalities A B]
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/precision_recall.py REAL GEN

Feature mode: REAL and GEN are ``.pt`` (a tensor) or ``.npy`` files of shape [N, K] (detector features, e.g. StyleGAN3's
VGG16 embeddings; K a multiple of 64).  Prints one JSON line (rank 0).

``--images``: REAL and GEN are images, embedded on the GPU by the VGG16 detector (DESIGN.md §13) with the torchvision
``vgg16`` weights of ``--vgg_state`` (a state_dict with ``features.*`` and ``classifier.*``).  Each is a reference image zip
(``ImgDataset``: entries of ``--split``, channels ``--modalities``, 0..255 mapped to [-1, 1]), an ``augment_dataset`` output
directory (its ``img_aug/img_aug_{i}`` pickles, modalities A and B), or a ``.pt`` tensor [N, C, H, W] in [-1, 1].  Prints one
JSON line per modality (rank 0).

Under torchrun every rank reads both inputs and the work is sharded by rows.
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


def load_images(path, split, modalities):
    """[N, C, H, W] fp32 in [-1, 1] on the host."""
    if path.endswith('.zip'):
        from latentaugment_b200.augments.utils.util_dataset import ImgDataset
        if not modalities:
            raise SystemExit(f'{path}: an image zip needs --modalities')
        ds = ImgDataset(path, split, modalities, resolution=None)
        return torch.stack([torch.from_numpy(ds[i][0] / 127.5 - 1) for i in range(len(ds))])
    if os.path.isdir(path):
        from latentaugment_b200.augments.utils.util_io import read_pickle
        d = os.path.join(path, 'img_aug')
        names = sorted((f for f in os.listdir(d) if f.startswith('img_aug_')), key=lambda f: int(f.rsplit('_', 1)[1]))
        if not names:
            raise SystemExit(f'{d}: no img_aug_{{i}} pickles')
        batches = [read_pickle(os.path.join(d, f)) for f in names]
        return torch.cat([torch.cat([torch.as_tensor(b['A']), torch.as_tensor(b['B'])], dim=1) for b in batches]).float()
    t = torch.load(path, map_location='cpu', weights_only=True)
    if not torch.is_tensor(t) or t.dim() != 4 or t.shape[2] != t.shape[3]:
        raise SystemExit(f'{path}: expected an [N, C, H, H] tensor')
    return t.float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('real')
    ap.add_argument('gen')
    ap.add_argument('--nhood', type=int, default=3)
    ap.add_argument('--images', action='store_true', help='REAL and GEN are images, embedded by the VGG16 detector')
    ap.add_argument('--vgg_state', help='torchvision vgg16 state_dict (--images)')
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32_parity'], help='detector precision (--images)')
    ap.add_argument('--split', default='train', help='split of an image zip (--images)')
    ap.add_argument('--modalities', nargs='+', help='channels of an image zip, in order (--images)')
    a = ap.parse_args()
    if a.images and not a.vgg_state:
        raise SystemExit('--images needs --vgg_state')
    rank, world, lr = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(lr)
    dev = torch.device(f'cuda:{lr}')
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    if a.images:
        images(a, rank, world, dev)
    else:
        features(a, rank, world, dev)
    if world > 1:
        dist.destroy_process_group()


def images(a, rank, world, dev):
    from latentaugment_b200.engine import FeatureDetector
    from latentaugment_b200.metrics import precision_recall_images
    real, gen = load_images(a.real, a.split, a.modalities), load_images(a.gen, a.split, a.modalities)
    if real.shape[1] != gen.shape[1]:
        raise SystemExit(f'REAL has {real.shape[1]} modalities, GEN {gen.shape[1]}')
    state = torch.load(a.vgg_state, map_location='cpu', weights_only=True)
    det = FeatureDetector(state, precision=a.precision, device=dev)
    for c in range(real.shape[1]):
        stats = {}
        p, r = precision_recall_images(det, real, gen, a.nhood, modality=c, stats=stats)
        if rank == 0:
            print(json.dumps({'modality': c, 'precision': p, 'recall': r, 'nhood_size': a.nhood, 'n_real': real.shape[0],
                              'n_gen': gen.shape[0], 'res_real': real.shape[2], 'res_gen': gen.shape[2], 'detector_precision': a.precision,
                              'n_gpus': world, **stats}))


def features(a, rank, world, dev):
    real, gen = load_features(a.real).to(dev), load_features(a.gen).to(dev)
    stats = {}
    p, r = precision_recall(real, gen, a.nhood, stats=stats)
    if rank == 0:
        print(json.dumps({'precision': p, 'recall': r, 'nhood_size': a.nhood, 'n_real': real.shape[0], 'n_gen': gen.shape[0],
                          'dim': real.shape[1], 'n_gpus': world, **stats}))


if __name__ == '__main__':
    main()
