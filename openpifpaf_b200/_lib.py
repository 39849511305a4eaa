"""ctypes binding of libpifpaf_b200.so (the C ABI declared in include/pifpaf_b200.h).

There is no CPU or eager fallback: if the shared library is missing or a call
fails (e.g. no B200 present) a RuntimeError is raised, like the reference's
TORCH_CHECK -> RuntimeError path (csrc/src/cifcaf.cpp:137-138).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'csrc', 'libpifpaf_b200.so')

OK, E_BADARG, E_CUDA, E_OVERFLOW, E_NOMEM = 0, 1, 2, 3, 4

c_i32, c_i64, c_f32, c_f64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_double
P = ctypes.POINTER
VP = ctypes.c_void_p


class DecoderParams(ctypes.Structure):
    """pifpaf_decoder_params_t"""
    _fields_ = [
        ('cifhr_neighbors', c_i64), ('cifhr_threshold', c_f64), ('cifhr_ablation_skip', c_i32),
        ('seed_threshold', c_f64), ('seeds_ablation_nms', c_i32), ('seeds_ablation_no_rescore', c_i32),
        ('caf_score_th', c_f64), ('caf_cif_floor', c_f64), ('caf_ablation_no_rescore', c_i32),
        ('block_joints', c_i32), ('greedy', c_i32),
        ('keypoint_threshold', c_f64), ('keypoint_threshold_rel', c_f64),
        ('reverse_match', c_i32), ('force_complete', c_i32), ('force_complete_caf_th', c_f64),
        ('nms_suppression', c_f64), ('nms_instance_threshold', c_f64), ('nms_keypoint_threshold', c_f64),
        ('occ_reduction', c_f64), ('occ_min_scale', c_f64), ('cifhr_revision', c_f64),
    ]


class CifDetParams(ctypes.Structure):
    """pifpaf_cifdet_params_t"""
    _fields_ = [
        ('cifhr_neighbors', c_i64), ('cifhr_threshold', c_f64), ('seed_threshold', c_f64),
        ('occ_reduction', c_f64), ('occ_min_scale', c_f64), ('cifhr_revision', c_f64),
        ('max_detections_before_nms', c_i64), ('nms', c_i32), ('nms_by_category', c_i32),
        ('iou_threshold', c_f64), ('suppression', c_f64), ('instance_threshold', c_f64),
    ]


# every symbol include/pifpaf_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    'pifpaf_last_error': (ctypes.c_char_p, []),
    'pifpaf_abi_version': (ctypes.c_int, []),
    'pifpaf_build_arch': (ctypes.c_char_p, []),
    'pifpaf_launch_count': (c_i64, []),
    'pifpaf_decoder_default_params': (ctypes.c_int, [P(DecoderParams)]),
    'pifpaf_decoder_create': (ctypes.c_int, [P(VP), c_i32, c_i32, c_i32, c_i32, VP,
                                             c_i32, c_i32, c_i32, c_i32, c_i32]),
    'pifpaf_decoder_destroy': (None, [VP]),
    'pifpaf_decoder_decode_device': (ctypes.c_int, [VP, VP, VP, c_i32, c_i32, c_i32, c_i32, c_i32,
                                                    VP, VP, VP, c_i32, P(DecoderParams), VP]),
    'pifpaf_decoder_fetch': (ctypes.c_int, [VP, VP, VP, VP, c_i32, VP]),
    'pifpaf_decoder_fetch_begin': (ctypes.c_int, [VP, VP]),
    'pifpaf_decoder_fetch_end': (ctypes.c_int, [VP, VP, VP, VP, c_i32]),
    'pifpaf_decoder_fetch_peek': (ctypes.c_int, [VP, VP]),
    'pifpaf_decoder_call': (ctypes.c_int, [VP, VP, c_i32, VP, c_i32, c_i32, c_i32, VP, VP, c_i32,
                                           P(DecoderParams), VP, VP, c_i32, P(c_i32)]),
    'pifpaf_decoder_tap_cifhr': (ctypes.c_int, [VP, c_i32, VP, c_i64]),
    'pifpaf_decoder_tap_seeds': (ctypes.c_int, [VP, c_i32, VP, VP, c_i64, P(c_i64)]),
    'pifpaf_decoder_tap_caf': (ctypes.c_int, [VP, c_i32, VP, VP, VP, VP]),
    'pifpaf_decoder_debug_set_epochs': (ctypes.c_int, [VP, ctypes.c_uint32, ctypes.c_uint32]),
    'pifpaf_decoder_last_stats': (ctypes.c_int, [VP, VP, c_i32]),
    'pifpaf_cifdet_default_params': (ctypes.c_int, [P(CifDetParams)]),
    'pifpaf_cifdet_create': (ctypes.c_int, [P(VP), c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32]),
    'pifpaf_cifdet_destroy': (None, [VP]),
    'pifpaf_cifdet_decode_device': (ctypes.c_int, [VP, VP, c_i32, c_i32, c_i32, c_i32, P(CifDetParams), VP]),
    'pifpaf_cifdet_fetch': (ctypes.c_int, [VP, VP, VP, c_i32, VP]),
    'pifpaf_cifdet_call': (ctypes.c_int, [VP, VP, c_i32, c_i32, c_i32, P(CifDetParams), VP, c_i32, P(c_i32)]),
    'pifpaf_image_resize_bilinear_u8': (ctypes.c_int, [VP, c_i32, c_i32, VP, c_i64, c_i32, c_i32, VP, VP, c_i32,
                                                        VP, VP, c_i32, VP, VP]),
    'pifpaf_image_fill_rgb': (ctypes.c_int, [VP, c_i64, c_i32, c_i32, c_i32, VP]),
    'pifpaf_net_create': (ctypes.c_int, [P(VP), c_i32, c_i32]),
    'pifpaf_net_destroy': (None, [VP]),
    'pifpaf_net_tensor': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, P(c_i32)]),
    'pifpaf_net_input_conv': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, VP, VP, c_i32, c_i32]),
    'pifpaf_net_conv1x1': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, c_i32, VP, VP, c_i32, c_i32, c_i32, c_i32, c_i32]),
    'pifpaf_net_conv1x1_scatter': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, c_i32, VP, VP, c_i32, c_i32, VP, VP, VP, VP]),
    'pifpaf_net_dw_conv1x1_scatter': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, VP, VP, c_i32,
                                                      c_i32, VP, VP, c_i32, c_i32, VP, VP, VP, VP]),
    'pifpaf_net_conv': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, VP, VP, c_i32, c_i32, c_i32,
                                       c_i32, c_i32]),
    'pifpaf_net_dwconv': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, VP, VP, c_i32, c_i32, c_i32]),
    'pifpaf_net_se_conv1x1': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, VP, VP, VP, VP, c_i32, VP, VP, c_i32, c_i32]),
    'pifpaf_net_heads': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, VP, VP, VP, VP, VP]),
    'pifpaf_net_heads_upsampled': (ctypes.c_int, [VP, c_i32, c_i32, c_i32, VP, VP, VP, c_i32, VP, VP]),
    'pifpaf_net_head_output': (ctypes.c_int, [VP, c_i32, P(VP), P(c_i32), P(c_i32), P(c_i32), P(c_i32)]),
    'pifpaf_net_set_head_buffers': (ctypes.c_int, [VP, c_i32]),
    'pifpaf_net_set_sm_limit': (ctypes.c_int, [VP, c_i32]),
    'pifpaf_net_forward': (ctypes.c_int, [VP, VP, c_i32, c_i32, VP]),
    'pifpaf_net_forward_u8': (ctypes.c_int, [VP, VP, c_i32, VP, VP, c_i32, VP]),
    'pifpaf_net_forward_timed': (ctypes.c_int, [VP, VP, c_i32, c_i32, VP, VP, VP, VP, VP]),
    'pifpaf_net_tap_tensor': (ctypes.c_int, [VP, c_i32, c_i32, VP, c_i64]),
    'pifpaf_net_set_tensor': (ctypes.c_int, [VP, c_i32, c_i32, VP, c_i64]),
    'pifpaf_net_flops_per_image': (c_f64, [VP]),
    'pifpaf_net_num_ops': (c_i32, [VP]),
    'pifpaf_grow_connection_blend': (ctypes.c_int, [VP, c_i64, c_f64, c_f64, c_f64, c_f64, c_i32, P(c_f64)]),
}

_lib = None


def lib():
    """Load libpifpaf_b200.so; raises RuntimeError (never falls back) if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                '(or make -C openpifpaf_b200/csrc). openpifpaf_b200 has no CPU fallback.')
        handle = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SYMBOLS.items():
            fn = getattr(handle, name)      # AttributeError if the export is missing
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def check(rc):
    if rc != OK:
        msg = lib().pifpaf_last_error().decode('utf-8', 'replace')
        raise RuntimeError(f'libpifpaf_b200 error {rc}: {msg}')


def default_params(**overrides):
    p = DecoderParams()
    check(lib().pifpaf_decoder_default_params(ctypes.byref(p)))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise AttributeError(f'unknown decoder parameter {k}')
        setattr(p, k, v)
    return p
