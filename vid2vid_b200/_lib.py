"""ctypes binding of libv2v_b200.so (C ABI declared in include/v2v_b200.h).

The library is built in-tree by vid2vid_b200/build.py (nvcc, sm_100a).  There is no CPU or
PyTorch fallback: if the shared object is missing or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('V2V_LIB') or os.path.join(_HERE, 'libv2v_b200.so')   # V2V_LIB: A/B timing of two builds

PAD_NONE, PAD_ZERO, PAD_REFLECT = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_LRELU, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3, 4
NORM_NONE, NORM_BATCH, NORM_INSTANCE = 0, 1, 2
IMPL_UMMA, IMPL_SIMT = 0, 1
PREC_BF16, PREC_BF16X3 = 0, 1


class ConvDesc(C.Structure):
    _fields_ = [('Cin', C.c_int), ('Cout', C.c_int), ('kh', C.c_int), ('kw', C.c_int), ('stride', C.c_int),
                ('pad', C.c_int), ('pad_mode', C.c_int), ('transposed', C.c_int), ('output_padding', C.c_int),
                ('weight', C.c_void_p), ('bias', C.c_void_p), ('Cout2', C.c_int), ('weight2', C.c_void_p),
                ('bias2', C.c_void_p)]


class NormDesc(C.Structure):
    _fields_ = [('kind', C.c_int), ('gamma', C.c_void_p), ('beta', C.c_void_p), ('running_mean', C.c_void_p),
                ('running_var', C.c_void_p), ('num_batches_tracked', C.c_void_p), ('momentum', C.c_float),
                ('eps', C.c_float)]


class HeadChannel(C.Structure):
    _fields_ = [('slot', C.c_int), ('channel', C.c_int), ('dst_C', C.c_int), ('act', C.c_int), ('scale', C.c_float)]


_lib = None
LAUNCHES = [0]      # kernels launched through this binding (bench.py's gpu_launches)

# every symbol include/v2v_b200.h declares (tests/test_host_logic.py checks the list against the header)
SYMBOLS = [
    'v2v_version', 'v2v_last_error',
    'v2v_correlation_out_shape', 'v2v_correlation_forward', 'v2v_resample2d_forward', 'v2v_channelnorm_forward',
    'v2v_resample_forward', 'v2v_onehot_edges', 'v2v_avgpool3s2', 'v2v_fg_mask',
    'v2v_face_window', 'v2v_crop_concat_forward', 'v2v_crop_backward',
    'v2v_l1_loss_forward', 'v2v_l1_loss_backward', 'v2v_mse_const_forward', 'v2v_mse_const_backward', 'v2v_avgpool3s2_backward',
    'v2v_resample_backward', 'v2v_ids_window_push', 'v2v_tensor2im_u8', 'v2v_flownet_prep', 'v2v_resize', 'v2v_sub_channels', 'v2v_flow_conf',
    'v2v_plan_create', 'v2v_plan_destroy', 'v2v_plan_set_precision', 'v2v_g_input', 'v2v_g_input_ex', 'v2v_g_conv', 'v2v_g_norm_act', 'v2v_g_norm_act_slice', 'v2v_g_conv_act',
    'v2v_g_head', 'v2v_g_concat', 'v2v_g_correlation', 'v2v_g_export', 'v2v_g_composite', 'v2v_g_composite_ex', 'v2v_plan_set_training', 'v2v_plan_backward', 'v2v_plan_finalize', 'v2v_plan_finalize_ws', 'v2v_plan_repack', 'v2v_plan_run',
    'v2v_plan_profile', 'v2v_plan_num_kernels', 'v2v_plan_conv_macs', 'v2v_plan_workspace_bytes', 'v2v_plan_describe',
    'v2v_conv_tap_table',
]


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError('libv2v_b200.so is not built (%s). Run `python -c "import __graft_entry__ as g; g.build()"` '
                           'or `python vid2vid_b200/build.py`. There is no fallback path.' % LIB_PATH)
    l = C.CDLL(LIB_PATH)
    l.v2v_last_error.restype = C.c_char_p
    l.v2v_plan_conv_macs.restype = C.c_double
    l.v2v_plan_workspace_bytes.restype = C.c_int64
    l.v2v_plan_describe.restype = C.c_int64
    l.v2v_plan_describe.argtypes = [C.c_void_p, C.c_char_p, C.c_int64]
    l.v2v_plan_create.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    l.v2v_plan_destroy.argtypes = [C.c_void_p]
    l.v2v_plan_set_precision.argtypes = [C.c_void_p, C.c_int]
    l.v2v_g_input.argtypes = [C.c_void_p] + [C.c_int] * 7 + [C.POINTER(C.c_int)]
    l.v2v_g_input_ex.argtypes = [C.c_void_p] + [C.c_int] * 8 + [C.POINTER(C.c_int)]
    l.v2v_g_conv.argtypes = [C.c_void_p, C.c_int, C.POINTER(ConvDesc), C.POINTER(C.c_int)]
    l.v2v_g_norm_act.argtypes = [C.c_void_p, C.c_int, C.POINTER(NormDesc), C.c_int, C.c_float, C.c_int, C.c_int,
                                 C.POINTER(C.c_int)]
    l.v2v_g_norm_act_slice.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(NormDesc), C.c_int, C.c_float, C.c_int,
                                       C.c_int, C.POINTER(C.c_int)]
    l.v2v_g_conv_act.argtypes = [C.c_void_p, C.c_int, C.POINTER(ConvDesc), C.c_int, C.c_float, C.POINTER(C.c_int)]
    l.v2v_g_head.argtypes = [C.c_void_p, C.c_int, C.POINTER(ConvDesc), C.POINTER(HeadChannel)]
    l.v2v_g_export.argtypes = [C.c_void_p, C.c_int, C.c_int]
    l.v2v_g_concat.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]
    l.v2v_g_correlation.argtypes = [C.c_void_p] + [C.c_int] * 8 + [C.c_float, C.POINTER(C.c_int)]
    l.v2v_g_composite.argtypes = [C.c_void_p] + [C.c_int] * 13
    l.v2v_plan_finalize.argtypes = [C.c_void_p, C.c_void_p]
    l.v2v_plan_finalize_ws.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    l.v2v_g_composite_ex.argtypes = [C.c_void_p] + [C.c_int] * 14
    l.v2v_plan_set_training.argtypes = [C.c_void_p, C.c_int]
    l.v2v_plan_backward.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p),
                                    C.POINTER(C.c_void_p), C.c_int, C.c_void_p]
    l.v2v_plan_repack.argtypes = [C.c_void_p, C.c_void_p]
    l.v2v_plan_run.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p]
    l.v2v_plan_profile.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int),
                                   C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int)]
    l.v2v_plan_num_kernels.argtypes = [C.c_void_p]
    l.v2v_plan_conv_macs.argtypes = [C.c_void_p]
    l.v2v_plan_workspace_bytes.argtypes = [C.c_void_p]
    fp, ip, vp = C.c_void_p, C.POINTER(C.c_int), C.c_void_p
    l.v2v_correlation_out_shape.argtypes = [C.c_int] * 7 + [ip, ip, ip]
    l.v2v_correlation_forward.argtypes = [fp, fp, fp] + [C.c_int] * 10 + [vp]
    l.v2v_resample2d_forward.argtypes = [fp, fp, fp] + [C.c_int] * 7 + [vp]
    l.v2v_channelnorm_forward.argtypes = [fp, fp] + [C.c_int] * 5 + [vp]
    l.v2v_resample_forward.argtypes = [fp, fp, fp] + [C.c_int] * 5 + [vp]
    l.v2v_onehot_edges.argtypes = [fp, fp, fp] + [C.c_int] * 5 + [vp]
    l.v2v_avgpool3s2.argtypes = [fp, fp] + [C.c_int] * 3 + [vp]
    l.v2v_fg_mask.argtypes = [fp, fp] + [C.c_int] * 6 + [ip, C.c_int, vp]
    l.v2v_l1_loss_forward.argtypes = [fp, fp, fp] + [C.c_int] * 4 + [vp, fp, vp]
    l.v2v_l1_loss_backward.argtypes = [fp, fp, fp] + [C.c_int] * 4 + [fp, fp, fp, vp]
    l.v2v_mse_const_forward.argtypes = [fp, C.c_int64, C.c_float, vp, fp, vp]
    l.v2v_mse_const_backward.argtypes = [fp, C.c_int64, C.c_float, fp, fp, vp]
    l.v2v_avgpool3s2_backward.argtypes = [fp, fp, C.c_int, C.c_int, C.c_int, vp]
    l.v2v_resample_backward.argtypes = [fp, fp, fp, fp, fp] + [C.c_int] * 5 + [vp]
    l.v2v_face_window.argtypes = [fp] + [C.c_int] * 7 + [vp, vp]
    l.v2v_crop_concat_forward.argtypes = [fp, C.c_int, fp] + [C.c_int] * 4 + [vp, C.c_int, C.c_int, fp, vp]
    l.v2v_crop_backward.argtypes = [fp] + [C.c_int] * 5 + [vp, C.c_int, C.c_int, fp, vp]
    l.v2v_ids_window_push.argtypes = [fp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    l.v2v_tensor2im_u8.argtypes = [fp, vp, C.c_int, C.c_int, C.c_int, vp]
    l.v2v_flownet_prep.argtypes = [fp, fp, C.c_int64, C.c_int64, fp, fp, fp, C.c_int, C.c_int, C.c_int, C.c_float, vp]
    l.v2v_resize.argtypes = [fp, fp, fp] + [C.c_int] * 7 + [C.c_float, C.c_float, C.c_float, vp]
    l.v2v_sub_channels.argtypes = [fp, fp, fp] + [C.c_int] * 6 + [vp]
    l.v2v_flow_conf.argtypes = [fp, fp, fp] + [C.c_int] * 4 + [C.c_float, vp]
    l.v2v_conv_tap_table.argtypes = [C.POINTER(ConvDesc), C.c_int, C.c_int, C.c_int] + [ip] * 15
    _lib = l
    return l


def check(rc):
    if rc != 0:
        msg = lib().v2v_last_error()
        raise RuntimeError('libv2v_b200: error %d: %s' % (rc, msg.decode() if msg else '?'))


def current_stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
