"""ctypes binding of libsfmloss.so (include/sfmloss.h).  No CPU fallback: a missing library or a
failing call raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libsfmloss.so')

SFM_MAX_SCALES = 4
SFM_MAX_SOURCES = 8
SFM_FLAG_TABLES_PROVIDED = 0x1
SFM_FLAG_REUSE_PYRAMID = 0x2
SFM_FLAG_NO_TMA = 0x4
SFM_FLAG_EDGE_AWARE_SMOOTH = 0x8
SFM_FLAG_IMAGE_GRADS = 0x10
SFM_FLAG_SNIPPET_TERMS = 0x20
SFM_FLAG_MIN_REPROJECTION = 0x40
SFM_FLAG_FULL_RES_MULTISCALE = 0x80
SFM_FLAG_MEAN_NORM_SMOOTH = 0x100
SFM_FLAG_EDGE_MEAN_ABS = 0x200
SFM_FLAG_BORDER_PADDING = 0x400
SFM_FLAG_AXISANGLE_POSE = 0x800
SFM_FLAG_GEOMETRY_CONSISTENCY = 0x1000
SFM_FLAG_POSE_INVERT_SHIFT = 16          # flags bit 16 + i: invert the transform of source i

SFM_E_INVALID_DESC = -1
SFM_E_INVALID_SHAPE = -2
SFM_E_NULL_POINTER = -3
SFM_E_UNSUPPORTED = -4
SFM_E_NO_DEVICE = -5
SFM_E_COMM = -6
SFM_NCCL_UNIQUE_ID_BYTES = 128
SFM_IPC_HANDLE_BYTES = 64

LOSS_KEYS = ('total_loss', 'pixel_loss', 'smooth_loss', 'exp_loss', 'ssim_loss')   # base_model.py:119-123

_vp = C.c_void_p


class SfmDesc(C.Structure):
    _fields_ = [('B', C.c_int32), ('S', C.c_int32), ('H', C.c_int32), ('W', C.c_int32),
                ('n_scales', C.c_int32), ('B_global', C.c_int32),
                ('smooth_reg', C.c_float), ('exp_reg', C.c_float), ('ssim_rate', C.c_float),
                ('flags', C.c_uint32), ('raw_disp_scales', C.c_uint32), ('raw_pose_hw', C.c_int32)]


class SfmInputs(C.Structure):
    _fields_ = [('tgt', _vp), ('src', _vp), ('intrinsics', _vp), ('disps', _vp * SFM_MAX_SCALES),
                ('poses', _vp), ('logits', _vp * SFM_MAX_SCALES), ('proj', _vp), ('kinv', _vp)]


class SfmGrads(C.Structure):
    _fields_ = [('gdisps', _vp * SFM_MAX_SCALES), ('gposes', _vp), ('glogits', _vp * SFM_MAX_SCALES)]


class SfmImageGrads(C.Structure):
    _fields_ = [('gtgt', _vp), ('gsrc', _vp)]


class SfmSnippetTerms(C.Structure):
    _fields_ = [('weights', _vp), ('losses', _vp)]


class SfmPixelTerms(C.Structure):
    _fields_ = [('weights', _vp * SFM_MAX_SCALES), ('losses', _vp * SFM_MAX_SCALES)]


class SfmMinReprojection(C.Structure):
    _fields_ = [('automask', C.c_int32), ('reserved_', C.c_int32), ('selection', _vp * SFM_MAX_SCALES)]


class SfmGeometry(C.Structure):
    _fields_ = [('src_disps', _vp * SFM_MAX_SCALES), ('gsrc_disps', _vp * SFM_MAX_SCALES),
                ('diff_maps', _vp * SFM_MAX_SCALES), ('geometry_reg', C.c_float), ('self_mask', C.c_int32)]


class SfmAugment(C.Structure):
    _fields_ = [('out_h', C.c_int32), ('out_w', C.c_int32), ('off_y', C.c_int32), ('off_x', C.c_int32),
                ('flip', C.c_int32), ('reserved_', C.c_int32), ('x_scaling', C.c_double), ('y_scaling', C.c_double)]


class SfmDebug(C.Structure):
    _fields_ = [('P', _vp * SFM_MAX_SCALES), ('u0', _vp * SFM_MAX_SCALES), ('v0', _vp * SFM_MAX_SCALES),
                ('inb', _vp * SFM_MAX_SCALES)]


# every symbol include/sfmloss.h declares: name -> (restype, argtypes)
_i = C.c_int
_D, _I, _G, _Dbg = C.POINTER(SfmDesc), C.POINTER(SfmInputs), C.POINTER(SfmGrads), C.POINTER(SfmDebug)
_IG = C.POINTER(SfmImageGrads)
_ST = C.POINTER(SfmSnippetTerms)
_PT = C.POINTER(SfmPixelTerms)
_MR = C.POINTER(SfmMinReprojection)
_GE = C.POINTER(SfmGeometry)
SYMBOLS = {
    'sfm_version': (_i, []),
    'sfm_last_error': (C.c_char_p, []),
    'sfm_workspace_bytes': (C.c_size_t, [_D]),
    'sfm_loss_forward': (_i, [_D, _I, _vp, _Dbg, _vp, _vp]),
    'sfm_loss_backward': (_i, [_D, _I, _vp, _G, _vp, _vp]),
    'sfm_loss_forward_backward': (_i, [_D, _I, _vp, _G, _vp, _vp]),
    'sfm_scale_grads': (_i, [_D, _vp, _G, _vp]),
    'sfm_loss_forward_backward_images': (_i, [_D, _I, _vp, _G, _IG, _vp, _vp]),
    'sfm_scale_image_grads': (_i, [_D, _vp, _IG, _vp]),
    'sfm_intrinsics_grad': (_i, [_D, _I, _vp, _vp, _vp]),
    'sfm_scale_intrinsics_grad': (_i, [_D, _vp, _vp, _vp]),
    'sfm_set_kernel_events': (_i, [_vp, _vp]),
    'sfm_pyramid': (_i, [_D, _vp, _vp, _vp, _vp]),
    'sfm_pyramid_export': (_i, [_D, _vp, _i, _vp, _vp, _vp]),
    'sfm_build_tables': (_i, [_D, _vp, _vp, _vp, _vp, _vp]),
    'sfm_ingest_u8': (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'sfm_eval_depth_scratch_bytes': (C.c_size_t, [_i, _i, _i]),
    'sfm_eval_depth': (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, C.c_float, C.c_float, _vp, _vp, _vp]),
    'sfm_disp_activation': (_i, [C.c_longlong, _vp, _vp, _vp, _vp]),
    'sfm_pose_reduce': (_i, [_i, _i, _i, _vp, _vp, _vp]),
    'sfm_upsample_disparity': (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp]),
    'sfm_warp_forward': (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'sfm_warp_backward_scratch_bytes': (C.c_size_t, [_i]),
    'sfm_warp_backward': (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'sfm_sampler_interp_forward': (_i, [_i] * 6 + [_vp, _vp, _vp, _vp]),
    'sfm_sampler_interp_backward': (_i, [_i] * 6 + [_vp, _vp, _vp, _vp, _vp, _vp]),
    'sfm_host_ctx_create': (_i, [_D, C.POINTER(_vp)]),
    'sfm_host_ctx_destroy': (_i, [_vp]),
    'sfm_loss_step_host': (_i, [_vp, _I, _vp, _G]),
    'sfm_loss_step_host_submit': (_i, [_vp, _I, _vp, _G]),
    'sfm_loss_step_host_wait': (_i, [_vp]),
    'sfm_loss_step_host_u8_submit': (_i, [_vp, _vp, _vp, _vp, _I, _vp, _G]),
    'sfm_nccl_set_library': (_i, [C.c_char_p]),
    'sfm_nccl_version': (_i, []),
    'sfm_comm_unique_id': (_i, [_vp]),
    'sfm_comm_create': (_i, [_vp, _i, _i, C.POINTER(_vp)]),
    'sfm_comm_destroy': (_i, [_vp]),
    'sfm_allreduce_partials': (_i, [_vp, _vp, _i, _vp]),
    'sfm_peer_create': (_i, [_i, _i, C.POINTER(_vp), _vp]),
    'sfm_peer_connect': (_i, [_vp, _vp]),
    'sfm_peer_destroy': (_i, [_vp]),
    'sfm_loss_forward_backward_peer': (_i, [_D, _I, _vp, _G, _vp, _vp, _vp]),
    'sfm_loss_snippets': (_i, [_D, _I, _ST, _vp, _G, _IG, _vp, _vp, _vp]),
    'sfm_loss_weighted': (_i, [_D, _I, _ST, _PT, _vp, _G, _IG, _vp, _vp, _vp]),
    'sfm_loss_min_reprojection': (_i, [_D, _I, _ST, _MR, _vp, _G, _vp, _vp, _vp]),
    'sfm_loss_geometry': (_i, [_D, _I, _ST, _GE, _vp, _G, _vp, _vp, _vp]),
}

_lib = None


class SfmError(RuntimeError):
    def __init__(self, code, msg):
        super(SfmError, self).__init__('libsfmloss error %d: %s' % (code, msg))
        self.code = code


def load():
    """Returns the loaded library; builds nothing and never falls back to CPU code."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError('%s is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                              '(there is no CPU fallback for the view-synthesis loss path)' % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise SfmError(rc, load().sfm_last_error().decode('utf-8', 'replace'))
