"""ctypes binding of libdt_b200.so (include/dt_b200.h, include/dt_b200_train3d.h).  No torch types cross
the boundary: tensors are passed as raw device pointers + sizes + stream."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libdt_b200.so')
_lib = None

_p = C.c_void_p
_i = C.c_int
_f = C.c_float
_sz = C.c_size_t

# name -> argtypes (every function returns int unless listed in _RESTYPE)
SIGNATURES = {
    'dt_abi_version': [],
    'dt_memset': [_p, _i, _sz, _p],
    'dt_pairs_to_f16': [_p, C.c_longlong, _i, _p, _p],
    'dt_scale_rois': [_p, _i, _i, _i, _p, _i, C.c_double, _p, _p],
    'dt_bbox_overlaps': [_p, _i, _i, _p, _i, _i, _i, _p, _i, _p],
    'dt_nms_workspace_bytes': [_i, _i, C.POINTER(_sz)],
    'dt_nms_batched': [_p, _i, _i, _i, _i, _p, _f, _i, _i, _i, _p, _p, _p, _sz, _p],
    'dt_lsa_batched': [_p, _i, _i, _i, _p, _p, _i, _p, _p, _p],
    'dt_match_frames': [_p, _i, _i, _i, _i, _p, _p, _f, _i, _p, _p, _p],
    'dt_assign_track_ids': [_p, _p, _p, _i, _i, _p, _i, _i, _i, _p, _p],
    'dt_pose_pck_cost': [_p, _i, _p, _i, _i, _i, _i, _i, _f, _p, _p],
    'dt_frame_costs': [_p, _i, _i, _p, _i, _i, _i, _i, _f, _p, _p, _i, _i, _f, C.c_double, _p, _p],
    'dt_prune_detections': [_p, _i, _i, _i, _i, _i, _p, _p, _f, _f, _p, _p, _p, _p],
    'dt_conv_plan': [C.c_void_p, _i, C.c_void_p],
    'dt_conv3d': [_p, _p, _p, _p, _p, _p, _p, _p],
    'dt_rpn_workspace_bytes': [_i, _i, C.POINTER(_i), C.POINTER(_i), _i, C.POINTER(_sz)],
    'dt_rpn_proposals_multi': [_p, _i, _i, _i, _i, _i, _p, _i, _f, C.c_double, C.c_longlong, _i, _i, _p, _sz, _p],
    'dt_collect_rpn': [_p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _i, _p],
    'dt_distribute_fpn': [_p, _i, _p, _i, _i, _i, _i, _i, _f, _f, _p, _p, _p, _p],
    'dt_box_decode': [_p, _p, _i, _i, _i, _p, _i, _p, _i, _i, _p, _p, C.POINTER(_f), C.c_double, _f, _p, _p, _p],
    'dt_limit_detections': [_p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _i, _p],
    'dt_prep_clip': [_p, _i, _i, _i, C.POINTER(_f), C.c_double, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    'dt_conv1_7x7s2': [_p, _i, _i, _i, _i, _p, _i, _p, _p, _i, _i, _i, _i, _i, _p, _i, _p],
    'dt_maxpool2d': [_p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p],
    'dt_roi_align': [C.POINTER(_p), C.POINTER(_i), C.POINTER(_i), C.POINTER(_f), _i, _i, _i, _i, _i, _p, _i, _p, _i,
                     _i, _p, _i, _i, _i, _i, _p, _p],
    'dt_keypoint_decode': [_p, _i, _i, _i, _i, _p, _i, _p, _i, _i, _p, _p, _p],
    'dt_conv1_7x7s2_f32': [_p, _i, _i, _i, _i, _p, _p, _p, _i, _p, _p],
    'dt_spatial_mean': [_p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p],
    'dt_time_mean': [_p, _i, _i, C.c_longlong, _i, _i, _i, _i, _i, _p, _i, _p],
    'dt_fold_tube_heads': [_p, _i, _i, _i, _i, _p, _p, _p],
    'dt_to_planes': [_p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    'dt_wgrad': [_p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    'dt_wgrad_nhwc': [_p, _i, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    'dt_bwd_pointwise': [_p, _p, _p, _p, C.c_longlong, _i, _p, _p],
    'dt_bwd_pointwise2': [_p, _p, _p, _p, C.c_longlong, _i, _p, _p, _p, _p],
    'dt_upsample_add_bwd': [_p, _p, _i, _i, _i, _i, _p, _p],
    'dt_scatter_stride2': [_p, _i, _i, _i, _i, _i, _i, _p, _p],
    'dt_sgd_update': [_p, _p, _p, _i, _i, _i, _f, _f, _f, _f, _p, _p, _p],
    'dt_sgd_update_multi': [_p, _p, _i, _i, _f, _f, _f, _f, _p],
    'dt_bias_grad': [_p, C.c_longlong, _i, _i, _p, _p],
    'dt_rpn_loss_grad': [_p, _i, _p, _p, _p, _p, C.c_longlong, _i, _f, _f, _f, _p, _i, _p, _p],
    'dt_embed_frame': [_p, _i, _i, C.c_longlong, _i, _p, _p],
    'dt_grad_join_f32': [_p, _p, C.c_longlong, _p, _p],
    'dt_roi_align_bwd': [_p, C.POINTER(_p), C.POINTER(_i), C.POINTER(_i), C.POINTER(_f), _i, _i, _i, _p, _i, _p, _i, _i, _p, _i, _i, _p],
    'dt_frcnn_loss_grad': [_p, _i, _p, _p, _p, _p, _i, _i, _p, _f, _f, _p, _i, _p, _p, _p],
    'dt_kps_loss_grad': [_p, _i, _i, _i, _i, _p, _p, _p, _f, _p, _i, _p, _p],
    'dt_subpixel_grad_fix': [_p, _p, _i, _i, _i, _p],
    'dt_jpeg_decode': [C.POINTER(C.c_char_p), C.POINTER(_sz), _i, _i, _i, _p, _p],
    'dt_rpn_targets_workspace_bytes': [_i, _i, C.POINTER(_i), C.POINTER(_i), _i, _i, C.POINTER(_sz)],
    'dt_rpn_targets': [_p, _i, _i, _i, _i, _p, _p, _p, _i, _p, _f, _f, _f, _i, _f, C.c_ulonglong, _p, _sz, _p],
    'dt_sample_rois': [_p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _i, _i, _i, _p, _i, _i, _f, _f, _f, _f, C.POINTER(_f), _i,
                       C.c_ulonglong, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _p, _p],
}
# the tube model's training-step entry points (include/dt_b200_train3d.h), error-code functions like the above
TRAIN3D_SIGNATURES = {
    'dt_rpn_tube_loss_grad': [_p, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _f, _f, _p, _p, _i, _p, _p],
    'dt_frcnn_tube_loss_grad': [_p, _i, _p, _p, _p, _p, _i, _i, _i, _p, _f, _f, _p, _i, _p, _p, _p],
    'dt_spatial_mean_bwd': [_p, C.c_longlong, _i, _i, _i, _p, _p, _p, _p, _p, _p],
}
# host-only helpers (not error-code functions)
HOST_FUNCS = {'dt_planes_ld': ([_i, _i, _i, _i], C.c_int), 'dt_jpeg_available': ([], C.c_int)}



class RpnLevel(C.Structure):
    """dt_rpn_level (include/dt_b200.h)."""
    _fields_ = [('logits', C.c_void_p), ('deltas', C.c_void_p), ('anchors', C.c_void_p), ('ld_s', C.c_int), ('ld_d', C.c_int),
                ('H', C.c_int), ('W', C.c_int), ('feat_stride', C.c_double), ('out', C.c_void_p), ('counts', C.c_void_p)]


class RpnTargetLevel(C.Structure):
    """dt_rpn_target_level (include/dt_b200.h)."""
    _fields_ = [('H', C.c_int), ('W', C.c_int), ('feat_stride', C.c_double), ('anchors', C.c_void_p), ('labels', C.c_void_p),
                ('bbox_targets', C.c_void_p), ('inside_weights', C.c_void_p), ('outside_weights', C.c_void_p),
                ('vis_labels', C.c_void_p)]


class SgdItem(C.Structure):
    """dt_sgd_item (include/dt_b200.h)."""
    _fields_ = [('w', C.c_void_p), ('g', C.c_void_p), ('m', C.c_void_p), ('w_fwd', C.c_void_p), ('w_dgrad', C.c_void_p),
                ('taps', C.c_int), ('Cout', C.c_int), ('Cin', C.c_int), ('tiles_ci', C.c_int), ('tiles_co', C.c_int),
                ('lr_mult', C.c_float), ('wd_mult', C.c_float)]


class ConvDesc(C.Structure):
    """dt_conv_desc (include/dt_b200.h)."""
    _fields_ = [(n, C.c_int) for n in (
        'N', 'Ti', 'Hi', 'Wi', 'Cin', 'Cout', 'kT', 'kH', 'kW', 'sT', 'sH', 'sW', 'pT', 'pH', 'pW',
        'in_ld', 'w_ld', 'out_ld', 'res_ld', 'dtype', 'out_f32', 'relu', 'res_mode', 'x3', 'in_lo_off', 'out_lo_off',
        'res_lo_off', 'out_round_tf32', 'out_time_major', 'out_t_first', 'out_t_count')]


class ConvPlan(C.Structure):
    """dt_conv_plan_t (include/dt_b200.h)."""
    _fields_ = [(n, C.c_int) for n in ('BN', 'TH', 'TW', 'TT', 'TB', 'tiles', 'kiters', 'stages', 'ks', 'ncbuf', 'nrbuf',
                                        'smem_bytes')] + [('useful_rows', C.c_double)]


_RESTYPE = {'dt_last_error': C.c_char_p}


def lib():
    """Load (once) and return the CDLL.  Raises RuntimeError if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                'libdt_b200.so is not built (%s). Run `python -m detectandtrack_b200.build` '
                '(or __graft_entry__.build()). There is no CPU fallback.' % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        l.dt_last_error.restype = C.c_char_p
        l.dt_last_error.argtypes = []
        for name, args in list(SIGNATURES.items()) + list(TRAIN3D_SIGNATURES.items()):
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = _RESTYPE.get(name, C.c_int)
        for name, (args, res) in HOST_FUNCS.items():
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = res
        _lib = l
    return _lib


def check(rc, what=''):
    if rc != 0:
        msg = lib().dt_last_error().decode('utf-8', 'replace')
        raise RuntimeError('%s failed (code %d): %s' % (what or 'libdt_b200 call', rc, msg))


def call(name, *args):
    check(getattr(lib(), name)(*args), name)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError('detectandtrack_b200 needs a CUDA device (B200, sm_100a); '
                           'there is no CPU fallback.')
    return torch


def ptr(t):
    """Device pointer of a (contiguous) torch tensor, or NULL for None."""
    if t is None:
        return None
    assert t.is_contiguous(), 'tensor must be contiguous'
    return C.c_void_p(t.data_ptr())


def zeros(shape, dtype):
    """torch.empty + dt_memset on the current stream: zero-initialised device tensor without a library kernel."""
    import torch
    t = torch.empty(shape, dtype=dtype, device='cuda')
    call('dt_memset', C.c_void_p(t.data_ptr()), 0, t.numel() * t.element_size(), stream_ptr())
    return t


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
