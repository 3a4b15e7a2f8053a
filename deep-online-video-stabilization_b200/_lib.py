"""ctypes loader of libmgw_b200.so -- the C ABI declared in include/mgw.h.

There is NO fallback: if the shared library is missing (and cannot be built because nvcc is absent) importing
this module raises, and every compute entry point returns an error without a CUDA device.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, os.environ.get('MGW_SO_NAME', 'libmgw_b200.so'))      # MGW_SO_NAME selects an A/B build (tuning only)

c_f = ctypes.c_void_p      # device pointers travel as raw addresses
c_i = ctypes.c_int
c_fl = ctypes.c_float
c_st = ctypes.c_void_p

# name -> (restype, argtypes); mirrors include/mgw.h one to one (tests/test_abi.py checks the header against this)
SIGNATURES = {
    'mgw_version': (c_i, []),
    'mgw_last_error': (ctypes.c_char_p, []),
    'mgw_launch_count': (ctypes.c_uint64, []),
    'mgw_vertices_fwd': (c_i, [c_f, c_i, c_i, c_i, c_fl, c_f, c_f, c_st]),
    'mgw_vertices_bwd': (c_i, [c_f, c_f, c_f, c_i, c_i, c_i, c_fl, c_f, c_st]),
    'mgw_solve_h_fwd': (c_i, [c_f, c_i, c_i, c_i, c_f, c_st]),
    'mgw_solve_h_bwd': (c_i, [c_f, c_f, c_f, c_i, c_i, c_i, c_f, c_st]),
    'mgw_warp_fwd': (c_i, [c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_f, c_st]),
    'mgw_warp_bwd_workspace_bytes': (ctypes.c_size_t, [c_i] * 6),
    'mgw_warp_bwd': (c_i, [c_f, c_f, c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_st]),
    'mgw_warp_bwd_acc': (c_i, [c_f, c_f, c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_st]),
    'mgw_mesh_warp_fwd': (c_i, [c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_f, c_st]),
    'mgw_mesh_warp_bwd_workspace_bytes': (ctypes.c_size_t, [c_i] * 6),
    'mgw_mesh_warp_bwd': (c_i, [c_f, c_f, c_f, c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_st]),
    'mgw_mesh_warp_bwd_acc': (c_i, [c_f, c_f, c_f, c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_st]),
    'mgw_mesh_warp_img_loss_fwd': (c_i, [c_f, c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_f, c_f, c_st]),
    'mgw_mesh_warp_img_loss_bwd_workspace_bytes': (ctypes.c_size_t, [c_i] * 6),
    'mgw_mesh_warp_img_loss_bwd': (c_i, [c_f] * 7 + [c_fl, c_f, c_fl, c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_st]),
    'mgw_feature_loss_dh': (c_i, [c_f] * 5 + [c_fl, c_f] + [c_i] * 6 + [c_f, c_st]),
    'mgw_loss_ratio_sum': (c_i, [c_f, c_i, c_i, c_fl, c_f, c_st]),
    'mgw_train_pass_fwd': (c_i, [c_f] * 7 + [c_i] * 7 + [c_fl] + [c_f] * 9 + [c_st]),
    'mgw_train_pass_bwd_workspace_bytes': (ctypes.c_size_t, [c_i] * 6),
    'mgw_train_pass_bwd': (c_i, [c_f] * 15 + [c_i] * 7 + [c_fl] + [c_f] * 3 + [c_st]),
    'mgw_remap_bundle_u8_workspace_bytes': (ctypes.c_size_t, [c_i, c_i, c_i]),
    'mgw_remap_bundle_u8': (c_i, [c_f, c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_resize_linear_u8': (c_i, [c_f, c_i, c_i, c_i, c_f, c_f, c_i, c_i, c_f, c_st]),
    'mgw_cvt_img2train_u8': (c_i, [c_f, c_i, c_i, c_f, c_f, c_f, c_i, c_f, c_f, c_f, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_warp_rev_bundle_u8': (c_i, [c_f, c_f, c_i, c_i, c_i, c_i, c_i, c_i, c_f, c_st]),
    'mgw_stream_assemble': (c_i, [c_f, c_f, c_i, c_i, ctypes.POINTER(ctypes.c_int), c_i, c_i, c_f, c_i, c_i, c_f, c_st]),
    'mgw_stream_push': (c_i, [c_f, c_f, c_i, c_i, c_f, c_f, c_i, c_i, c_f, c_i, c_st]),
    'mgw_vertex_losses_fwd': (c_i, [c_f, c_f, c_f, c_i, c_i, c_i, c_fl, c_f, c_f, c_st]),
    'mgw_vertex_losses_bwd': (c_i, [c_f, c_f, c_f, c_i, c_i, c_i, c_fl, c_f, c_f, c_f, c_f, c_st]),
    'mgw_u8_to_train_f32': (c_i, [c_f, c_f, ctypes.c_size_t, c_st]),
    'mgw_train_f32_to_u8': (c_i, [c_f, c_f, ctypes.c_size_t, c_st]),
    'mgw_fill_zero': (c_i, [c_f, ctypes.c_size_t, c_i, c_st]),
    'mgw_black_accumulate': (c_i, [c_f, c_f, c_i, c_st]),
    'mgw_crop_rect_workspace_bytes': (ctypes.c_size_t, [c_i, c_i]),
    'mgw_crop_rect': (c_i, [c_f, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_stream_assemble_dev': (c_i, [c_f, c_f, c_i, c_f, ctypes.POINTER(ctypes.c_int), c_i, c_i, c_f, c_i, c_i, c_f, c_st]),
    'mgw_stream_push_dev': (c_i, [c_f, c_f, c_i, c_f, c_f, c_f, c_i, c_i, c_st]),
    'mgw_cvt_img2train_u8_batch': (c_i, [c_f, c_i, c_i, c_i, c_f, c_f, c_f, c_i, c_f, c_f, c_f, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_resize_linear_u8_batch': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_i, c_i, c_f, c_st]),
    'mgw_streams_assemble': (c_i, [c_f, c_f, c_i, c_i, c_f, ctypes.POINTER(ctypes.c_int), c_i, c_i, c_f, c_i, c_i, c_f, c_st]),
    'mgw_streams_push': (c_i, [c_f, c_f, c_i, c_i, c_f, c_f, c_f, c_i, c_i, c_st]),
    'mgw_cvt_img2train_yuv420_batch': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_f, c_i, c_f, c_f, c_f, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_resize_linear_yuv420_batch': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_i, c_i, c_f, c_st]),
    'mgw_cvt_img2train_mixed': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_f, c_f, c_i, c_f, c_f, c_f, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_resize_linear_mixed': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_f, c_i, c_i, c_f, c_st]),
    'mgw_remap_bundle_frame_workspace_bytes': (ctypes.c_size_t, [c_i] * 5),
    'mgw_remap_bundle_frame': (c_i, [c_f, c_i, c_f, c_i, c_i, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_remap_bundle_frame_yuv420': (c_i, [c_f, c_i, c_f, c_i, c_i, c_i, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_remap_bundle_frame_mixed': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_copy_slots_mixed': (c_i, [c_f, c_f, c_i, c_i, c_i, c_i, c_f, c_st]),
    'mgw_cvt_img2train_planes': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_f, c_i, c_f, c_f, c_f, c_i, c_i, c_i, c_f, c_f, c_st]),
    'mgw_resize_linear_planes': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_i, c_i, c_f, c_st]),
    'mgw_remap_bundle_frame_planes': (c_i, [c_f, c_i, c_f, c_i, c_i, c_i, c_i, c_i, c_f, c_i, c_f, c_st]),
    'mgw_cvt_img2train_mixed_planes': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_f, c_f, c_i, c_f, c_f, c_f, c_i, c_i, c_i, c_f, c_f,
                                             c_st]),
    'mgw_resize_linear_mixed_planes': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_f, c_i, c_i, c_f, c_st]),
    'mgw_remap_bundle_frame_mixed_planes': (c_i, [c_f, c_i, c_i, c_i, c_i, c_f, c_f, c_i, c_i, c_f, c_i, c_f, c_st]),
    'mgw_interp_fwd': (c_i, [c_f, c_f, c_f] + [c_i] * 6 + [c_f, c_st]),
    'mgw_interp_bwd': (c_i, [c_f, c_f, c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_st]),
    'mgw_homography_warp_fwd': (c_i, [c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_f, c_st]),
    'mgw_homography_warp_bwd': (c_i, [c_f, c_f, c_f] + [c_i] * 6 + [c_f, c_f, c_st]),
    'mgw_img_loss_fwd': (c_i, [c_f, c_f, c_f] + [c_i] * 4 + [c_f, c_st]),
    'mgw_img_loss_bwd': (c_i, [c_f, c_f, c_f, c_f, c_fl, c_f] + [c_i] * 4 + [c_f, c_st]),
    'mgw_feature_loss_fwd': (c_i, [c_f, c_f, c_f] + [c_i] * 4 + [c_f, c_f, c_st]),
    'mgw_feature_loss_bwd': (c_i, [c_f, c_f, c_f, c_fl, c_f] + [c_i] * 4 + [c_f, c_st]),
    'mgw_temp_loss_fwd': (c_i, [c_f] * 5 + [c_i] * 4 + [c_f, c_st]),
    'mgw_temp_loss_bwd': (c_i, [c_f] * 6 + [c_fl, c_f] + [c_i] * 4 + [c_f, c_f, c_st]),
}


class mgw_planes(ctypes.Structure):
    """include/mgw.h's mgw_planes: one frame's plane addresses (plane[0] == 0: the slot is idle) and row pitches in bytes"""
    _fields_ = [('plane', ctypes.c_uint64 * 3), ('pitch', ctypes.c_int32 * 3), ('reserved', ctypes.c_int32 * 3)]


class MgwError(RuntimeError):
    pass


def _load():
    if not os.path.exists(SO):
        try:
            from . import build as _build
            _build.build()
        except Exception as e:      # noqa: BLE001
            raise ImportError('libmgw_b200.so is missing and could not be built (%s). Run '
                              '`python __graft_entry__.py build`; there is no CPU fallback.' % e) from e
    lib = ctypes.CDLL(SO)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)     # AttributeError here = the .so does not match include/mgw.h
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(rc, what):
    if rc != 0:
        raise MgwError('%s failed (%d): %s' % (what, rc, lib.mgw_last_error().decode()))


def launch_count():
    return int(lib.mgw_launch_count())


def set_impl(mode):
    """'auto' (pipeline / TMA tiles when the shape allows, else generic) | 'generic' | 'tma' (one TMA tile per CTA, error if the
    shape does not fit) | 'pipe' (the persistent forward pipeline, the backward as 'tma'; error if the shape does not fit)"""
    if mode not in ('auto', 'generic', 'tma', 'pipe'):
        raise ValueError('unknown kernel family %r' % (mode,))
    os.environ['MGW_IMPL'] = mode          # the library reads the variable at every call: a test / tuning hook, not an ABI entry
