"""Output side of the caller loop (reference ``backbone_latentaug.py:91-124`` + ``utils/util_io.py:64-71``): every batch
leaves four pickles -- the input dict, the input latents, the augmented dict, the augmented latents -- under
``{outdir}/{img,latent,img_aug,latent_aug}/`` with ``pickle.HIGHEST_PROTOCOL``, same names and dict layouts, so whatever
reads the reference's output directory reads this one.

What changes is WHEN the files are written: ``AsyncPickleWriter`` serialises and writes on a worker thread, and
``augment_dataset`` drives ``LatentAugment.iterate`` (one batch of look-ahead), so pickling and disk time of batch t overlap
the kernels of batch t+1 instead of sitting between two batches (SURVEY.md §8f rank 4).
"""
import os
import pickle
import queue
import threading
import zipfile

import numpy as np
import torch

OUT_DIRS = ('img', 'latent', 'img_aug', 'latent_aug')       # backbone_latentaug.py:73


def write_pickle(data, path):
    """util_io.py:64-66"""
    with open(path, 'wb') as handle:
        pickle.dump(data, handle, protocol=pickle.HIGHEST_PROTOCOL)


def read_pickle(path):
    """util_io.py:68-71 (trusted files only: this is plain ``pickle.load``, as in the reference)."""
    with open(path, 'rb') as handle:
        return pickle.load(handle)


def _own(obj):
    """Deep copy of the tensors in a (nested) dict / list: the plugin's output dicts are views of pinned staging buffers
    that are reused two batches later; the writer thread must not race with that."""
    if isinstance(obj, torch.Tensor):
        return obj.detach().clone()
    if isinstance(obj, np.ndarray):
        return obj.copy()
    if isinstance(obj, dict):
        return {k: _own(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return type(obj)(_own(v) for v in obj)
    return obj


class AsyncPickleWriter:
    """``submit(obj, path)`` returns at once; a worker thread pickles and writes in submission order.  At most
    ``max_pending`` objects wait (``submit`` blocks beyond that, so memory stays bounded); ``close()`` drains the queue and
    re-raises the first error of the worker."""

    def __init__(self, max_pending=8):
        self._q = queue.Queue(maxsize=max_pending)
        self._err = None
        self.written = 0
        self._t = threading.Thread(target=self._run, name='latentaugment-writer', daemon=True)
        self._t.start()

    def _run(self):
        while True:
            item = self._q.get()
            try:
                if item is None:
                    return
                if self._err is None:
                    write_pickle(*item)
                    self.written += 1
            except Exception as exc:      # noqa: BLE001 -- reported by close() / the next submit()
                self._err = exc
            finally:
                self._q.task_done()

    def submit(self, obj, path, copy=True):
        if self._err is not None:
            raise self._err
        self._q.put((_own(obj) if copy else obj, path))

    def close(self):
        self._q.put(None)
        self._t.join()
        if self._err is not None:
            raise self._err

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


def augment_dataset(augment, dataset, outdir, n_iter=None, writer=None, verbose=True):
    """The reference's inner loop (backbone_latentaug.py:91-124) over ``dataset`` (an iterable of batch dicts): for batch i
    writes ``img/img_{i}``, ``latent/w_{i}``, ``img_aug/img_aug_{i}``, ``latent_aug/w_aug_{i}`` -- each only if its directory
    exists, as the reference does -- through the look-ahead loop and an asynchronous writer.  Returns the number of batches."""
    own_writer = writer is None
    writer = writer or AsyncPickleWriter()
    have = {d: os.path.exists(os.path.join(outdir, d)) for d in OUT_DIRS}

    def limited():
        for i, data in enumerate(dataset):
            if n_iter is not None and i >= n_iter:
                break
            yield data
    n = 0
    try:
        for i, (data, data_aug, data_w, data_w_aug) in enumerate(augment.iterate(limited(), with_latents=True)):
            if verbose:
                print(f'Iteration: {i} of {n_iter}')
            if have['img']:
                writer.submit(data, os.path.join(outdir, 'img', f'img_{i}'))
            if have['latent'] and data_w is not None:          # (None: the batch passed through un-augmented, p_thres)
                writer.submit(data_w, os.path.join(outdir, 'latent', f'w_{i}'))
            if have['img_aug']:
                writer.submit(data_aug, os.path.join(outdir, 'img_aug', f'img_aug_{i}'))
            if have['latent_aug'] and data_w_aug is not None:
                writer.submit(data_w_aug, os.path.join(outdir, 'latent_aug', f'w_aug_{i}'))
            n += 1
    finally:
        if own_writer:
            writer.close()
    return n


def invert_dataset(engine, img_zip, out_zip, *, split, modalities, num_steps=1000, seed=0, verbose=False, **project_kw):
    """Projects every image of ``img_zip`` (``ImgDataset`` layout: one pickled dict of 0..255 slices per entry; entries of
    ``split`` -- one name or a list, all written into the one zip --, channels = ``modalities`` in order) into W and writes
    ``out_zip``: the same entry names, each a pickled
    float32 ndarray ``[num_ws, w_dim]`` (the code broadcast to every layer) -- the ``{dataset_w_name}.zip`` that
    ``LatentCodeDataset`` / ``banks_from_reference_layout`` read for ``--init_w inv``.

    ``engine``: a ``SynthesisEngine`` with ``set_lpips(..., per_sample_targets=True)`` done.  Images are mapped to
    ``x / 127.5 - 1`` and projected ``engine.batch`` at a time (batch i with ``seed + i``); the last batch is padded by
    repeating its last image and the padded rows are dropped (rows are independent, so padding changes no code).
    Returns the number of codes written."""
    from .util_dataset import ImgDataset
    splits = [split] if isinstance(split, str) else list(split)
    B = engine.batch
    os.makedirs(os.path.dirname(os.path.abspath(out_zip)), exist_ok=True)
    tmp = out_zip + '.partial'
    total, bi = 0, 0
    with zipfile.ZipFile(tmp, 'w', zipfile.ZIP_STORED) as zf:
        for sp in splits:
            ds = ImgDataset(img_zip, split=sp, modalities=modalities, resolution=engine.img_resolution)
            names = ds.fnames
            for i0 in range(0, len(names), B):
                rows = list(range(i0, min(i0 + B, len(names))))
                x = np.stack([ds[r][0] for r in rows] + [ds[rows[-1]][0]] * (B - len(rows)))
                engine.set_projection_targets(torch.from_numpy(x) / 127.5 - 1)
                w = engine.project(num_steps=num_steps, seed=seed + bi, **project_kw)
                w = w.detach().float().cpu().numpy()
                for k, r in enumerate(rows):
                    code = np.repeat(w[k:k + 1], engine.num_ws, axis=0).astype('float32')
                    zf.writestr(names[r], pickle.dumps(code, protocol=pickle.HIGHEST_PROTOCOL))
                bi += 1
                if verbose:
                    print(f'{sp}: projected {rows[-1] + 1} / {len(names)}')
            total += len(names)
    os.replace(tmp, out_zip)
    return total
