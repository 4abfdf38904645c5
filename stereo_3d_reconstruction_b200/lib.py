# -*- coding: utf-8 -*-
"""ctypes binding of libs3d_b200.so (C ABI declared in include/s3d.h).

The library is the product's only compute path.  There is no CPU or PyTorch fallback: if the
shared object is missing, or a compute entry point is called without a CUDA device, this module
raises -- it never silently computes something else.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('S3D_LIB_PATH') or os.path.join(_HERE, 'libs3d_b200.so')   # env override: A/B-testing builds

S3D_MAX_TAPS = 64
DTYPE_F32, DTYPE_BF16, DTYPE_BF16X2 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_LEAKY, ACT_SIGMOID, ACT_TANH = 0, 1, 2, 3, 4


class S3dConvParams(ctypes.Structure):
    """Mirror of `struct S3dConvParams` (include/s3d.h)."""
    _fields_ = [
        ('N', ctypes.c_int32), ('iD', ctypes.c_int32), ('iH', ctypes.c_int32), ('iW', ctypes.c_int32),
        ('Cin', ctypes.c_int32),
        ('oD', ctypes.c_int32), ('oH', ctypes.c_int32), ('oW', ctypes.c_int32), ('Cout', ctypes.c_int32),
        ('sz', ctypes.c_int32), ('sy', ctypes.c_int32), ('sx', ctypes.c_int32),
        ('ntaps', ctypes.c_int32), ('n_classes', ctypes.c_int32),
        ('dz', ctypes.c_int8 * S3D_MAX_TAPS), ('dy', ctypes.c_int8 * S3D_MAX_TAPS),
        ('dx', ctypes.c_int8 * S3D_MAX_TAPS),
        ('osN', ctypes.c_int64), ('osD', ctypes.c_int64), ('osH', ctypes.c_int64), ('osW', ctypes.c_int64),
        ('osC', ctypes.c_int64),
        ('os_lo', ctypes.c_int64),
        ('omz', ctypes.c_int32), ('omy', ctypes.c_int32), ('omx', ctypes.c_int32),
        ('cout_store', ctypes.c_int32),
        ('in_dtype', ctypes.c_int32), ('out_dtype', ctypes.c_int32),
        ('act', ctypes.c_int32), ('act_param', ctypes.c_float),
        ('tw', ctypes.c_int32), ('th', ctypes.c_int32), ('td', ctypes.c_int32), ('tn', ctypes.c_int32),
        ('bn', ctypes.c_int32),
        ('proj_w', ctypes.c_void_p), ('proj_channel', ctypes.c_int32), ('proj_act', ctypes.c_int32),
        ('w_nstack', ctypes.c_void_p),
        ('dz_nref', ctypes.c_int32), ('dz_c', ctypes.c_int32), ('dz_e', ctypes.c_int32), ('dz_pairs', ctypes.c_int32),
        ('dz_sched', ctypes.c_void_p), ('dz_planes', ctypes.c_void_p),
    ]


_vp, _i, _f, _i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_int64
_CONV_SIG = [ctypes.POINTER(S3dConvParams), _vp, _vp, _vp, _vp, _vp, _vp]

# name -> argtypes; must list every symbol include/s3d.h declares (checked by tests/test_abi.py)
SIGNATURES = {
    's3d_version': ([], ctypes.c_char_p),
    's3d_last_error': ([], ctypes.c_char_p),
    's3d_device_check': ([_i], _i),
    's3d_set_knob': ([ctypes.c_char_p, _i], _i),
    's3d_get_knob': ([ctypes.c_char_p], _i),
    's3d_conv_igemm': (_CONV_SIG, _i),
    's3d_conv_direct': (_CONV_SIG, _i),
    's3d_pack_image': ([_vp, _vp, _f, _vp, _i, _i, _i, _i, _i, _vp], _i),
    's3d_pack_image_u8': ([_vp, _vp, _f, _f, _vp, _i, _i, _i, _i, _i, _vp], _i),
    's3d_conv_first': ([_vp, _i, _vp, _f, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp], _i),
    's3d_conv_concat_volume': ([ctypes.POINTER(S3dConvParams), _vp, _i, _i, _vp, _vp, _vp], _i),
    's3d_conv_concat_volume_ro': ([ctypes.POINTER(S3dConvParams), _vp, _i, _i, _vp, _vp, _vp, _vp], _i),
    's3d_conv_cls_workspace_bytes': ([_i, _i, _i, _i], ctypes.c_int64),
    's3d_conv_cls_soft_argmin': ([ctypes.POINTER(S3dConvParams), _vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_float, _vp], _i),
    's3d_conv2d_halo': ([_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i64, _i64, _i64, _i, _vp], _i),
    's3d_map_conv': ([_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp], _i),
    's3d_concat_gonce_assemble': ([_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp], _i),
    's3d_cost_volume_concat': ([_vp, _vp, _i, _i, _i, _i, _i, _i, _vp], _i),
    's3d_soft_argmin': ([_vp, _vp, _i, _i, _i, _i, _f, _vp], _i),
    's3d_tap_gather_soft_argmin': ([_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp], _i),
    's3d_cls_soft_argmin': ([_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp], _i),
    's3d_corr_soft_argmin': ([_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp], _i),
    's3d_upsample_disp': ([_vp, _vp, _i, _i, _i, _i, _i, _f, _vp], _i),
    's3d_upsample_disp_eval': ([_vp, _vp, _i, _i, _i, _i, _i, _f,
                                _vp, ctypes.POINTER(_f), _i, _f, _vp,
                                _vp, _f, _vp,
                                _vp, _vp, ctypes.POINTER(_f), _i, _vp, _vp], _i),
    's3d_disp_cloud_workspace_bytes': ([_i, _i], ctypes.c_int64),
    's3d_disp_cloud': ([_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _f, _vp, _f, _vp, _vp, _vp, _vp, _i64, _vp], _i),
    's3d_speckle_filter_workspace_bytes': ([_i, _i, _i], ctypes.c_int64),
    's3d_speckle_filter': ([_vp, _i, _i, _i, _vp, _i, _f, _vp, ctypes.POINTER(_f), _i, _f, _vp, _vp, _vp, _i64, _vp], _i),
    's3d_disp_wls_workspace_bytes': ([_i, _i, _i], ctypes.c_int64),
    's3d_disp_wls': ([_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _f, _vp, ctypes.POINTER(_f), _i, _f, _vp, _vp, _vp, _i64, _vp],
                     _i),
    's3d_latent_to_vox': ([_vp, _vp, _i, _i, _i, _i, _i, _i, _vp], _i),
    's3d_avg_pool': ([_vp, _vp, _i, _i, _i, _i, _i, _i, _vp], _i),
    's3d_depth_to_space': ([_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp], _i),
    's3d_split_tf32': ([_vp, _vp, _vp, _i64, _vp], _i),
    's3d_split_bf16': ([_vp, _vp, _i64, _i, _vp], _i),
    's3d_unsplit_bf16': ([_vp, _vp, _i64, _i, _vp], _i),
    's3d_fuse_views': ([_vp, _i64, _vp, _i64, _i, _vp, _i, _i, _i, _vp, ctypes.POINTER(_f), _i, _vp, _i64, _i64, _vp], _i),
    's3d_voxel_surface_workspace_bytes': ([_i, _i, _i], ctypes.c_int64),
    's3d_voxel_surface_eval': ([_vp, _vp, _i, _i, ctypes.POINTER(_f), _i, ctypes.POINTER(_i), _i, _vp, _vp, _i64, _vp], _i),
    's3d_voxel_surface_eval_hist': ([_vp, _vp, _i, _i, ctypes.POINTER(_f), _i, ctypes.POINTER(_i), _i, _vp, _vp, _i64, _vp,
                                     ctypes.POINTER(_i), _i, _vp], _i),
    's3d_voxel_mesh_bounds': ([_i, ctypes.POINTER(_i), ctypes.POINTER(_i)], _i),
    's3d_voxel_mesh': ([_vp, _i, _i, _f, _vp, _i, _vp, _i, _vp, _vp], _i),
    's3d_occupancy_curves': ([_vp, _vp, _i, _i, _i, _vp, _vp, _vp], _i),
    's3d_chamfer_forward': ([_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp], _i),
    's3d_chamfer_workspace_bytes': ([_i, _i, _i], ctypes.c_int64),
    's3d_chamfer_forward_ws': ([_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i64, _vp], _i),
    's3d_chamfer_eval': ([_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, ctypes.POINTER(_f), _i, _vp, _vp, _i64, _vp], _i),
    's3d_chamfer_eval_hist': ([_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, ctypes.POINTER(_f), _i, _vp, _vp, _i64, _vp,
                               ctypes.POINTER(_f), _i, _vp], _i),
    's3d_fma_probe': ([_vp, _i, ctypes.POINTER(ctypes.c_int64), _vp], _i),
}

_lib = None


class S3dError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises S3dError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise S3dError(
            'libs3d_b200.so not found at %s -- build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(or `make -C stereo_3d_reconstruction_b200/csrc`).  There is no CPU fallback.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (argtypes, restype) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().s3d_last_error().decode('utf-8', 'replace')
        raise S3dError('%s failed (rc=%d): %s' % (what, rc, msg))


# ---- A/B knobs ---------------------------------------------------------------------------------------------------
# Read ONCE (here, at import) from the S3D_* environment variables, never on the forward path.  The host-side ones live
# in this dict; the launcher-side ones live in the library (include/s3d.h, s3d_set_knob).  set_knob() changes either
# at run time (tests, A/B scripts) -- a model picks host-side knobs up at its next pack().
HOST_KNOBS = ('no_vol2d', 'no_concat_fuse', 'no_cls_fused', 'no_conv_first', 'no_d2s', 'no_ref_once', 'no_cls_chain', 'no_sheared', 'no_map_conv', 'no_conv2d_halo')
LIB_KNOBS = ('no_scatter', 'scatter_tps3', 'scatter_no_pair', 'scatter_ring', 'scatter_res_transpose',
             'scatter_no_transpose', 'scatter_generic', 'no_corr_tc', 'scatter_zsplit', 'scatter_no_rm', 'igemm_ts1', 'igemm_one_cta', 'scatter_one_cta', 'no_conv_first_tc', 'chamfer_sym', 'chamfer_sym_r', 'no_dz_skip')
KNOBS = {k: int(os.environ.get('S3D_' + k.upper()) is not None) for k in HOST_KNOBS}
KNOBS['no_scatter'] = int(os.environ.get('S3D_NO_SCATTER') is not None)        # both sides look at this one


def set_knob(name, value):
    value = int(value)
    if name in LIB_KNOBS:
        check(load().s3d_set_knob(name.encode(), value), 's3d_set_knob')
    elif name not in HOST_KNOBS:
        raise KeyError('unknown knob %r' % name)
    if name in KNOBS:
        KNOBS[name] = value


_launches = 0


def count_launch(n=1):
    """Bookkeeping for bench.py's `gpu_launches`: every kernel this package enqueues is counted."""
    global _launches
    _launches += n


def launches():
    return _launches
