"""ctypes binding of ``include/latentaugment_b200.h`` (the C-ABI shared library).

There is NO fallback: if the library is missing or a kernel fails, the call raises.
"""
import ctypes as C
import os

from . import _build

LA_MAX_BLOCKS = 12
LA_MAX_CONV = 2 * LA_MAX_BLOCKS
LA_MAX_MAPPING = 8
LA_MAX_STEPS = 64
LA_LOSS_COLS = 5
LA_VGG_CONVS, LA_VGG_TAPS = 13, 5
ABI_VERSION = 203          # == LA_ABI_VERSION of include/latentaugment_b200.h
PRECISION = {'bf16': 0, 'fp32_parity': 1}
NOISE = {'none': 0, 'const': 1, 'random': 2}

fptr = C.c_void_p


class ConvParams(C.Structure):
    _fields_ = [('d_weight', fptr), ('d_bias', fptr), ('d_noise_const', fptr), ('noise_strength', C.c_float),
                ('d_affine_weight', fptr), ('d_affine_bias', fptr)]


class ToRgbParams(C.Structure):
    _fields_ = [('d_weight', fptr), ('d_bias', fptr), ('d_affine_weight', fptr), ('d_affine_bias', fptr)]


class GeneratorDesc(C.Structure):
    _fields_ = [('img_resolution', C.c_int), ('img_channels', C.c_int), ('w_dim', C.c_int), ('z_dim', C.c_int),
                ('num_blocks', C.c_int), ('channels', C.c_int * LA_MAX_BLOCKS), ('conv_clamp', C.c_float),
                ('d_const', fptr), ('d_resample_filter', fptr),
                ('conv', ConvParams * LA_MAX_CONV), ('torgb', ToRgbParams * LA_MAX_BLOCKS),
                ('mapping_layers', C.c_int), ('mapping_lr_multiplier', C.c_float),
                ('d_mapping_weight', fptr * LA_MAX_MAPPING), ('d_mapping_bias', fptr * LA_MAX_MAPPING),
                ('d_w_avg', fptr)]


class AugmentOptions(C.Structure):
    _fields_ = [('num_steps', C.c_int), ('lr', C.c_float), ('w_latent', C.c_float), ('w_pix', C.c_float),
                ('soft_aug', C.c_int), ('alpha', C.c_float), ('final_noise_mode', C.c_int), ('n_modalities', C.c_int),
                ('w_disc', C.c_float), ('w_lpips', C.c_float), ('lpips_crop_x', C.c_int), ('lpips_crop_y', C.c_int),
                ('lpips_norm_mode', C.c_int)]


class VggDesc(C.Structure):
    _fields_ = [('d_conv_weight', fptr * LA_VGG_CONVS), ('d_conv_bias', fptr * LA_VGG_CONVS), ('d_lin_weight', fptr * LA_VGG_TAPS),
                ('mean', C.c_float * 3), ('std', C.c_float * 3), ('crop_size', C.c_int), ('per_sample_targets', C.c_int)]


class DetectorDesc(C.Structure):
    _fields_ = [('d_conv_weight', fptr * LA_VGG_CONVS), ('d_conv_bias', fptr * LA_VGG_CONVS), ('d_fc6_weight', fptr), ('d_fc6_bias', fptr),
                ('d_fc7_weight', fptr), ('d_fc7_bias', fptr), ('mean', C.c_float * 3), ('std', C.c_float * 3)]


class DiscBlockParams(C.Structure):
    _fields_ = [('d_fromrgb_weight', fptr), ('d_fromrgb_bias', fptr), ('d_conv0_weight', fptr), ('d_conv0_bias', fptr),
                ('d_conv1_weight', fptr), ('d_conv1_bias', fptr), ('d_skip_weight', fptr)]


class DiscDesc(C.Structure):
    _fields_ = [('img_resolution', C.c_int), ('img_channels', C.c_int), ('num_blocks', C.c_int),
                ('channels', C.c_int * LA_MAX_BLOCKS), ('conv_clamp', C.c_float), ('mbstd_group_size', C.c_int),
                ('d_resample_filter', fptr), ('block', DiscBlockParams * LA_MAX_BLOCKS),
                ('d_b4_conv_weight', fptr), ('d_b4_conv_bias', fptr), ('d_b4_fc_weight', fptr), ('d_b4_fc_bias', fptr),
                ('d_b4_out_weight', fptr), ('d_b4_out_bias', fptr)]


# name -> (restype, argtypes); every symbol include/latentaugment_b200.h declares
SIGNATURES = {
    'la_last_error': (C.c_char_p, []),
    'la_version': (C.c_int, []),
    'la_struct_sizes': (C.c_int, [C.POINTER(C.c_size_t), C.c_int]),
    'la_engine_workspace_bytes': (C.c_int, [C.POINTER(GeneratorDesc), C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    'la_engine_create': (C.c_int, [C.POINTER(GeneratorDesc), C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                   C.POINTER(C.c_void_p)]),
    'la_engine_destroy': (None, [C.c_void_p]),
    'la_set_latent_bank': (C.c_int, [C.c_void_p, fptr, C.c_int, C.c_void_p]),
    'la_set_image_bank': (C.c_int, [C.c_void_p, fptr, C.c_int, C.c_void_p]),
    'la_mapping': (C.c_int, [C.c_void_p, fptr, C.c_int, C.c_float, fptr, C.c_void_p]),
    'la_synthesis': (C.c_int, [C.c_void_p, fptr, C.c_longlong, C.c_longlong, C.c_int, fptr, fptr, C.c_void_p]),
    'la_noise_floats': (C.c_size_t, [C.c_void_p]),
    'la_augment': (C.c_int, [C.c_void_p, fptr, C.POINTER(AugmentOptions), fptr, fptr, fptr, fptr, C.c_void_p]),
    'la_disc_workspace_bytes': (C.c_int, [C.POINTER(DiscDesc), C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    'la_set_discriminator': (C.c_int, [C.c_void_p, C.POINTER(DiscDesc), C.c_void_p, C.c_size_t, C.c_void_p]),
    'la_disc_logits': (C.c_int, [C.c_void_p, fptr, fptr, C.c_void_p]),
    'la_disc_loss_grad': (C.c_int, [C.c_void_p, fptr, C.c_float, fptr, fptr, C.c_void_p]),
    'la_lpips_workspace_bytes': (C.c_int, [C.POINTER(VggDesc), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    'la_set_lpips': (C.c_int, [C.c_void_p, C.POINTER(VggDesc), C.c_void_p, C.c_size_t, C.c_void_p]),
    'la_set_feature_bank': (C.c_int, [C.c_void_p, fptr, C.c_int, C.c_void_p]),
    'la_lpips_loss_grad': (C.c_int, [C.c_void_p, fptr, C.c_int, C.c_int, C.c_float, C.c_int, fptr, fptr, C.c_void_p]),
    'la_lpips_tap': (C.c_int, [C.c_void_p, C.c_int, fptr, C.POINTER(C.c_size_t), C.c_void_p]),
    'la_set_projection_targets': (C.c_int, [C.c_void_p, fptr, C.c_void_p]),
    'la_project': (C.c_int, [C.c_void_p, fptr, C.c_int, fptr, fptr, fptr, fptr, fptr, C.c_void_p]),
    'la_filtered_lrelu': (C.c_int, [fptr, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_float), C.c_int,
                                    fptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int,
                                    C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, fptr, C.c_void_p]),
    'la_pairwise_sqdist': (C.c_int, [fptr, C.c_int, fptr, C.c_int, C.c_int, fptr, C.c_void_p]),
    'la_bank_prepare': (C.c_int, [fptr, C.c_int, C.c_int, C.c_void_p, fptr, C.c_void_p]),
    'la_nearest_codes': (C.c_int, [fptr, C.c_int, fptr, C.c_void_p, fptr, C.c_int, C.c_int, C.c_int, C.c_longlong,
                                   C.c_void_p, C.c_size_t, fptr, C.c_void_p, C.c_void_p]),
    'la_nearest_codes_workspace_bytes': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    'la_merge_topk': (C.c_int, [fptr, C.c_void_p, C.c_int, C.c_int, C.c_int, fptr, C.c_void_p, C.c_void_p]),
    'la_merge_topk_strided': (C.c_int, [fptr, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_longlong, fptr, C.c_void_p,
                                        C.c_void_p]),
    'la_pr_manifold_prepare': (C.c_int, [fptr, C.c_int, C.c_int, C.c_void_p, fptr, C.c_void_p]),
    'la_pr_radii_workspace_bytes': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    'la_pr_radii': (C.c_int, [fptr, C.c_int, fptr, C.c_void_p, fptr, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, fptr,
                              C.c_void_p, C.c_void_p]),
    'la_pr_member_workspace_bytes': (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    'la_pr_member': (C.c_int, [fptr, C.c_int, fptr, C.c_void_p, fptr, fptr, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                               C.c_void_p, C.c_void_p]),
    'la_detector_workspace_bytes': (C.c_int, [C.POINTER(DetectorDesc), C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    'la_detector_create': (C.c_int, [C.POINTER(DetectorDesc), C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_void_p)]),
    'la_detector_destroy': (None, [C.c_void_p]),
    'la_detector_features': (C.c_int, [C.c_void_p, fptr, C.c_int, C.c_int, C.c_int, C.c_int, fptr, C.c_void_p]),
    'la_debug_set_simt':(C.c_int, [C.c_void_p, C.c_int]),
    'la_debug_launch_count': (C.c_longlong, [C.c_void_p]),
    'la_debug_get': (C.c_int, [C.c_void_p, C.c_int, fptr, C.POINTER(C.c_size_t), C.c_void_p]),
    'la_debug_check': (C.c_int, [C.c_void_p, C.c_void_p]),
    'la_debug_time_gemms': (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
}

_lib = None


class LatentAugmentError(RuntimeError):
    pass


def lib_path():
    return _build.LIB


def load():
    """Loads ``liblatentaugment_b200.so`` (building it in-tree with nvcc if it is stale and
    nvcc is present).  Raises if it cannot be had -- there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    _build.build(force=os.environ.get('LA_REBUILD') == '1')     # content-hashed and incremental: a no-op when current
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    # the structs passed by pointer must have the layout the library was compiled with
    if lib.la_version() != ABI_VERSION:
        raise LatentAugmentError(f'{path} has ABI version {lib.la_version()}, the Python binding expects {ABI_VERSION}: '
                                 'rebuild with `python -m latentaugment_b200._build --force`')
    sizes = (C.c_size_t * 8)()
    n = lib.la_struct_sizes(sizes, 8)
    mine = [C.sizeof(t) for t in (GeneratorDesc, AugmentOptions, DiscDesc, ConvParams, ToRgbParams, DiscBlockParams, VggDesc, DetectorDesc)]
    if n < len(mine) or list(sizes)[:len(mine)] != mine:
        raise LatentAugmentError(f'struct layout mismatch between {path} {list(sizes)[:n]} and the ctypes binding {mine}')
    _lib = lib
    return lib


def check(code):
    if code != 0:
        msg = load().la_last_error()
        raise LatentAugmentError(f'latentaugment_b200 error {code}: {msg.decode() if msg else "?"}')
