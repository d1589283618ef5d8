"""Projects the real images of an image zip into W and writes the inverted-code zip ``--init_w inv`` reads.

    python tools/invert_dataset.py --interim_dir DIR --generator_state G.pt --vgg_state vgg.pt [--split train]

Reads ``{interim_dir}/{dataset_aug}/{dataset_name_aug}.zip`` (or ``--img_zip``) and writes
``{interim_dir}/{dataset_aug}/{dataset_w_name}.zip`` (or ``--out``), so ``create_augment`` with the same ``--interim_dir``
finds the codes.  The generator comes from ``--generator_state`` or from the reference's ``--model_dir`` tree; the VGG16 +
LPIPS parameters from ``--vgg_state`` with all five lin layers (``lin.0`` .. ``lin.4``).  See DESIGN.md "Projection".
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

TAPS = (4, 9, 16, 23, 30)


def _clamp(v):
    return None if str(v).lower() == 'none' else float(v)


def parse(argv=None):
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument('--model_dir', default='')
    p.add_argument('--interim_dir', default='')
    p.add_argument('--dataset_aug', default='Pelvis_2.1_repo_no_mask')
    p.add_argument('--dataset_name_aug', default='Pelvis_2.1_repo_no_mask-num-375_train-0.70_val-0.20_test-0.10')
    p.add_argument('--dataset_w_name', default='Pelvis_2.1_repo_no_mask-num-375_train-0.70_val-0.20_test-0.10-expinv_00001')
    p.add_argument('--modalities_aug', default='MR_nonrigid_CT,MR_MR_T2')
    p.add_argument('--exp_stylegan', default='00003')
    p.add_argument('--network_pkl_stylegan', default='network-snapshot-005320.pkl')
    p.add_argument('--generator_state', default='', help='torch state_dict file with the reference parameter names')
    p.add_argument('--vgg_state', default='', help='VGG16 (features.*) + LPIPS lin.0 .. lin.4 state_dict file')
    p.add_argument('--img_zip', default='', help='image zip (default: {interim_dir}/{dataset_aug}/{dataset_name_aug}.zip)')
    p.add_argument('--out', default='', help='code zip (default: {interim_dir}/{dataset_aug}/{dataset_w_name}.zip)')
    p.add_argument('--split', default='train', help='comma-separated splits, all written into the one --out zip (entry names '
                   'carry their split, as in the reference\'s zips); inverting one split at a time into the default --out overwrites it')
    p.add_argument('--conv_clamp', type=_clamp, default=256.0, help='generator conv_clamp with --generator_state (a number or none; '
                   'use the value create_augment will run with); a --model_dir network pickle brings its own')
    p.add_argument('--precision', default='fp32_parity', choices=['fp32_parity', 'bf16'])
    p.add_argument('--batch', type=int, default=32)
    p.add_argument('--num_steps', type=int, default=1000)
    p.add_argument('--seed', type=int, default=0)
    p.add_argument('--gpu', type=int, default=0)
    return p.parse_args(argv)


def main(argv=None):
    args = parse(argv)
    from latentaugment_b200.augments.utils import util_io
    from latentaugment_b200.augments.utils.util_latent_aug import load_stylegan_states, reference_network_pickle_path
    from latentaugment_b200.engine import SynthesisEngine
    from latentaugment_b200.utils import synthetic
    root = os.path.join(args.interim_dir, args.dataset_aug)
    img_zip = args.img_zip or os.path.join(root, args.dataset_name_aug + '.zip')
    out = args.out or os.path.join(root, args.dataset_w_name + '.zip')
    conv_clamp = args.conv_clamp
    if args.generator_state:
        G = torch.load(args.generator_state, map_location='cpu', weights_only=True)
    else:
        pkl = reference_network_pickle_path(args)
        if pkl is None:
            sys.exit('no generator: pass --generator_state FILE or --model_dir with the reference\'s network pickle')
        G, _, net_kw = load_stylegan_states(pkl)
        conv_clamp = net_kw.get('conv_clamp', conv_clamp)
    if not args.vgg_state:
        sys.exit('--vgg_state FILE is required (VGG16 + the five LPIPS lin layers)')
    vgg = torch.load(args.vgg_state, map_location='cpu', weights_only=True)
    kw = synthetic.infer_generator_kwargs(G)
    res = kw['img_resolution']
    eng = SynthesisEngine(G, batch=args.batch, precision=args.precision, device=f'cuda:{args.gpu}', conv_clamp=conv_clamp, **kw)
    eng.set_lpips(vgg, taps=TAPS, crop_size=min(res, 256), per_sample_targets=True)
    mods = [m for m in args.modalities_aug.split(',') if m]
    t0 = time.time()
    splits = [s for s in args.split.split(',') if s]
    n = util_io.invert_dataset(eng, img_zip, out, split=splits, modalities=mods, num_steps=args.num_steps, seed=args.seed,
                               verbose=True)
    print(f'wrote {n} codes to {out} in {time.time() - t0:.1f} s')


if __name__ == '__main__':
    main()
