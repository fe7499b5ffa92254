"""ctypes binding of libgen6d_b200.so (include/gen6d_b200.h).

The product path has NO fallback: if the library is missing or a call fails, an exception is
raised.  `lib()` loads lazily so that importing the package (parameter containers, host
geometry) works on machines without the built library; any compute call needs it.
"""
import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libgen6d_b200.so')
HEADER_PATH = os.path.join(os.path.dirname(HERE), 'include', 'gen6d_b200.h')

G6D_DET_MAX_SCALES = 8
PRO_NONE, PRO_AFFINE, PRO_AFFINE_RELU, PRO_CORR = 0, 1, 2, 3
ACT_NONE, ACT_RELU, ACT_LEAKY01 = 0, 1, 2
TC_TF32, TC_F16 = 0, 1


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ('B', 'D', 'H', 'W', 'Cin', 'in_cstride', 'in_coff', 'Cout', 'kd', 'kh', 'kw',
                                       'stride', 'pd', 'ph', 'pw', 'Do', 'Ho', 'Wo', 'out_cstride', 'out_coff',
                                       'prologue')] + [('group_rows', C.c_longlong), ('act', C.c_int), ('max_chain_k', C.c_int),
                                                           ('in_items', C.c_int)]


class DetMaps(C.Structure):
    _fields_ = [('n_scales', C.c_int), ('rfn', C.c_int), ('hs', C.c_int), ('ws', C.c_int),
                ('map', (C.c_void_p * 3) * G6D_DET_MAX_SCALES),
                ('H', (C.c_int * 3) * G6D_DET_MAX_SCALES), ('W', (C.c_int * 3) * G6D_DET_MAX_SCALES),
                ('mu', C.c_float * 3), ('inv_sigma', C.c_float * 3), ('clip', C.c_float)]


class GlueCamera(C.Structure):        # g6d_glue_camera (20 doubles: a float64 [qn, 20] numpy array has this layout)
    _fields_ = [('K', C.c_double * 9), ('Kinv', C.c_double * 9), ('f', C.c_double), ('f_sq', C.c_double)]


class GlueRefs(C.Structure):          # g6d_glue_refs
    _fields_ = [('poses', C.c_void_p), ('cen', C.c_void_p), ('f', C.c_void_p), ('dist', C.c_void_p), ('center', C.c_double * 3)]


class GlueViews(C.Structure):         # g6d_glue_views
    _fields_ = [('poses', C.c_void_p), ('R_look', C.c_void_p), ('RlookR', C.c_void_p), ('f', C.c_void_p), ('Kinv', C.c_void_p),
                ('src', C.c_void_p), ('rows', C.c_void_p), ('cols', C.c_void_p), ('even_idx', C.c_void_p), ('even_dirs', C.c_void_p),
                ('n_views', C.c_int), ('n_even', C.c_int), ('ref_num', C.c_int), ('size', C.c_int),
                ('norm_scale', C.c_double), ('norm_offset', C.c_float * 3), ('size_scale', C.c_float)]


P, I, L, F = C.c_void_p, C.c_int, C.c_longlong, C.c_float
_SIGNATURES = {
    'g6d_preprocess_u8': [P, P, L, I, I, P],
    'g6d_imagenet_norm': [P, P, L, I, I, P],
    'g6d_warp_perspective_u8': [P, I, P, I, I, P],
    'g6d_warp_affine_u8': [P, I, P, I, I, P],
    'g6d_glue_detection_jobs': [P, P, I, I, I, I, P, P],
    'g6d_glue_detection_jobs_host': [P, P, I, I, I, I, P],
    'g6d_glue_initial_poses': [P, P, P, C.POINTER(GlueRefs), P, I, P, P],
    'g6d_glue_initial_poses_host': [P, P, P, C.POINTER(GlueRefs), P, I, P],
    'g6d_glue_refine_problems': [C.POINTER(GlueViews), P, P, I, I, P, I, I, P, P, P, P, P, P, P, P],
    'g6d_glue_refine_problems_host': [C.POINTER(GlueViews), P, P, I, I, P, I, I, P, P, P, P, P, P, P],
    'g6d_glue_apply_refinements': [C.POINTER(GlueViews), P, P, P, P, I, P, P],
    'g6d_glue_apply_refinements_host': [C.POINTER(GlueViews), P, P, P, P, I, P],
    'g6d_track_smooth': [P, P, P, P, P, I, I, P, P, P, P, P, P],
    'g6d_track_smooth_host': [P, P, P, P, P, I, I, P, P, P, P, P],
    'g6d_nchw_to_nhwc': [P, P, I, I, I, I, I, P],
    'g6d_nhwc_to_nchw': [P, P, I, I, I, I, I, P],
    'g6d_resize_bilinear': [P, P, I, I, I, I, I, I, I, I, P],
    'g6d_resize_nearest': [P, P, I, I, I, I, I, I, P],
    'g6d_maxpool2x2': [P, P, I, I, I, I, P],
    'g6d_l2norm_channels': [P, P, L, I, F, P],
    'g6d_affine_act': [P, P, L, I, L, P, P, I, I, I, I, I, P],
    'g6d_avgpool_affine': [P, P, L, I, I, L, P, P, I, P],
    'g6d_add': [P, P, P, L, P],
    'g6d_instnorm_stats': [P, L, I, I, I, L, F, P, P, P, P],
    'g6d_instnorm_partial': [P, L, I, I, I, L, P, P],
    'g6d_instnorm_finalize': [P, L, I, L, F, P, P, P],
    'g6d_conv': [C.POINTER(ConvDesc), P, P, P, P, P, P, P, P],
    'g6d_conv_workspace_bytes': [C.POINTER(ConvDesc)],
    'g6d_vgg_first_block': [P, P, P, P, I, I, I, P],
    'g6d_pack_conv_weight': [P, P, I, I, I, I, P, P],
    'g6d_conv_tc_supported': [C.POINTER(ConvDesc), I],
    'g6d_conv_tc_debug': [C.POINTER(C.c_int)],
    'g6d_debug_umma_shift': [P, I, I, P],
    'g6d_conv_tc_workspace_bytes': [C.POINTER(ConvDesc), I],
    'g6d_conv_tc': [C.POINTER(ConvDesc), P, P, P, I, I, P, P, P, P, P, P, L, P],
    'g6d_conv_tc_stats_supported': [C.POINTER(ConvDesc), I, L],
    'g6d_pack_conv_weight_tc': [P, P, P, I, I, I, I, I, P, I, P],
    'g6d_split_operand': [P, P, P, L, I, P],
    'g6d_transpose2d': [P, P, I, I, P],
    'g6d_linear_smallm': [P, P, P, P, I, I, I, I, P],
    'g6d_det_score_fuse': [C.POINTER(DetMaps), I, P, P, P, P, P, P],
    'g6d_det_parse': [P, P, P, I, I, I, I, P, P, P],
    'g6d_det_corr_rowsum': [P, P, I, I, I, I, I, P],
    'g6d_sel_ref_sums': [P, I, I, I, P, P, P],
    'g6d_sel_corr_prologue': [P, P, P, I, I, I, I, F, P, P, P],
    'g6d_sel_corr_score': [P, P, I, I, I, P, P],
    'g6d_sel_corr_score3': [P, P, P, P, P, P, I, I, I, I, I, I, P, P, P, P],
    'g6d_sel_corr_score3_workspace_bytes': [I, I, I, I, I],
    'g6d_sel_vp_norm': [P, I, I, I, F, P, I, I, P],
    'g6d_sel_max_angle_add': [P, P, P, I, I, I, I, P],
    'g6d_attention': [P, P, P, P, I, I, I, I, P],
    'g6d_attention_headmajor': [P, P, P, P, I, I, I, I, P],
    'g6d_layernorm': [P, P, P, P, I, I, F, P],
    'g6d_sel_parse': [P, P, I, I, P, P, P],
    'g6d_ref_volume_fill': [P, P, P, P, P, P, I, I, I, I, I, I, I, I, P, P, P],
    'g6d_ref_pose_heads': [P, P, P, P, I, I, P],
    'g6d_pose_errors_workspace_bytes': [I, I],
    'g6d_pose_errors': [P, I, P, P, P, I, I, P, P, P],
}
_RESTYPE = {'g6d_pose_errors_workspace_bytes': L, 'g6d_sel_corr_score3_workspace_bytes': L, 'g6d_conv_workspace_bytes': L, 'g6d_conv_tc_workspace_bytes': L, 'g6d_launch_count': L, 'g6d_last_error': C.c_char_p}

_lib = None


class Gen6DLibraryError(RuntimeError):
    pass


def header_symbols():
    """Every function name declared in include/gen6d_b200.h."""
    text = open(HEADER_PATH).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(g6d_[a-z0-9_]+)\s*\(', text)))


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise Gen6DLibraryError(
            f'{LIB_PATH} not found: build it with `python -m gen6d_b200.build` '
            '(there is no CPU or PyTorch fallback for the Gen6D hot path)')
    l = C.CDLL(LIB_PATH)
    for name, args in _SIGNATURES.items():
        fn = getattr(l, name)
        fn.argtypes = args
        fn.restype = _RESTYPE.get(name, I)
    l.g6d_last_error.restype = C.c_char_p
    l.g6d_last_error.argtypes = []
    l.g6d_version.restype = I
    l.g6d_launch_count.restype = L
    _lib = l
    return l


def check(rc, name):
    if rc != 0:
        msg = lib().g6d_last_error().decode(errors='replace')
        raise Gen6DLibraryError(f'{name} failed ({rc}): {msg}')


def launch_count():
    return int(lib().g6d_launch_count())
