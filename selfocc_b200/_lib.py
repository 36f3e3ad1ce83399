"""ctypes binding of libselfocc_b200.so (the C ABI in include/selfocc_b200.h).

There is NO fallback: if the shared library is missing or an entry point is absent this module
raises, and every op in ``selfocc_b200.ops`` raises when handed a non-CUDA tensor.
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('SELFOCC_B200_LIB') or os.path.join(_PKG, 'lib', 'libselfocc_b200.so')   # env: experimental variant
ABI_VERSION = 5


class AxisMap(C.Structure):
    _fields_ = [('start', C.c_float), ('range0', C.c_float), ('range1', C.c_float), ('size0', C.c_float),
                ('size1', C.c_float), ('offset', C.c_float)]


class VolumeDesc(C.Structure):
    _fields_ = [('H', C.c_int32), ('W', C.c_int32), ('Z', C.c_int32), ('zpitch', C.c_int32),
                ('n_feat', C.c_int32), ('feat_pitch', C.c_int32), ('axis', AxisMap * 3)]


class RayDesc(C.Structure):
    _fields_ = [('n_cam', C.c_int32), ('rays_per_cam', C.c_int32), ('nx', C.c_int32), ('ny', C.c_int32),
                ('sx', C.c_float), ('ox', C.c_float), ('sy', C.c_float), ('oy', C.c_float),
                ('ray_begin', C.c_int64), ('ray_count', C.c_int64), ('chunk_len', C.c_int64)]


class OccGrid(C.Structure):
    _fields_ = [('n0', C.c_int32), ('n1', C.c_int32), ('n2', C.c_int32), ('z_lo', C.c_int32), ('z_hi', C.c_int32),
                ('border', C.c_int32 * 4), ('thresh', C.c_float)]


class ReprojDesc(C.Structure):
    _fields_ = [('variant', C.c_int32), ('n_cam', C.c_int32), ('n_rays', C.c_int32), ('n_samples', C.c_int32),
                ('img_h', C.c_int32), ('img_w', C.c_int32), ('size_h', C.c_float), ('size_w', C.c_float),
                ('grid_h', C.c_int32), ('grid_w', C.c_int32), ('ssim', C.c_int32), ('automask', C.c_int32)]


REPROJ_COMBINE, REPROJ_MONO_MULTI_NEW = 0, 1


class RenderParams(C.Structure):
    _fields_ = [('aabb', C.c_float * 6), ('near_plane', C.c_float), ('training', C.c_int32),
                ('num_samples', C.c_int32), ('inv_s', C.c_float), ('cos_anneal', C.c_float),
                ('anchor_mid', C.c_int32), ('sh_act', C.c_int32), ('bkgd_mode', C.c_int32)]


_P = C.c_void_p
_I = C.c_int32
_L = C.c_int64
_F = C.c_float

# name -> (restype, argtypes); must list every symbol declared in include/selfocc_b200.h
SIGNATURES = {
    'so_abi_version': (C.c_int, []),
    'so_last_cuda_error': (C.c_int, []),
    'so_error_string': (C.c_char_p, [C.c_int]),
    'so_launch_count': (C.c_int64, []),
    'so_profile_enable': (C.c_int, [C.c_int]),
    'so_profile_reset': (C.c_int, []),
    'so_profile_elapsed_ms': (C.c_int, [C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
    'so_tpv_decode': (C.c_int, [_P, _P, _P, _I, _P, _P, _P, _P, C.POINTER(VolumeDesc), _P, _P, _P]),
    'so_tpv_decode_rows': (C.c_int, [_P, _P, _P, _I, _P, _P, _P, _P, C.POINTER(VolumeDesc), _I, _I, _P, _P, _P]),
    'so_tpv_decode_bwd_features': (C.c_int, [_P, _P, _P, _I, C.POINTER(VolumeDesc), _I, _I, _P, _P]),
    'so_tpv_decode_bwd_hidden': (C.c_int, [_P, _P, _P, _P, _I, C.POINTER(VolumeDesc), _I, _I, _P, _P, _P]),
    'so_tpv_decode_bwd_input': (C.c_int, [_P, _P, _L, _P]),
    'so_tpv_decode_force_simt': (C.c_int, [C.c_int]),
    'so_render_train_force_fwd32': (C.c_int, [C.c_int]),
    'so_render_train_force_sem_generic': (C.c_int, [C.c_int]),
    'so_render_workspace_floats': (C.c_int64, [_L]),
    'so_render_infer': (C.c_int, [_P, _P, C.POINTER(VolumeDesc), _P, _P, C.POINTER(RayDesc), C.POINTER(RenderParams),
                                  _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'so_render_pack_floats': (_L, [C.POINTER(VolumeDesc)]),
    'so_render_pack': (C.c_int, [_P, _P, C.POINTER(VolumeDesc), _P, _P]),
    'so_render_infer_packed': (C.c_int, [_P, _P, C.POINTER(VolumeDesc), _P, _P, _P, C.POINTER(RayDesc), C.POINTER(RenderParams),
                                         _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'so_render_train_forward': (C.c_int, [_P, _P, C.POINTER(VolumeDesc), _P, _P, C.POINTER(RayDesc), C.POINTER(RenderParams),
                                          _P, _P] + [_P] * 11 + [_P, _P, _P]),
    'so_render_train_pair_floats': (_L, [C.POINTER(VolumeDesc)]),
    'so_render_train_backward': (C.c_int, [_P, _P, C.POINTER(VolumeDesc), _P, _P, C.POINTER(RayDesc), C.POINTER(RenderParams),
                                           _P, _P] + [_P] * 7 + [_P, _P, _P, _P, _P]),
    'so_field_query_backward': (C.c_int, [C.POINTER(VolumeDesc), _P, _L, _P, _P, _P, _P, _P, _P]),
    'so_field_second_grad': (C.c_int, [_P, C.POINTER(VolumeDesc), _P, _L, _P, _P]),
    'so_field_second_grad_backward': (C.c_int, [C.POINTER(VolumeDesc), _P, _L, _P, _P, _P]),
    'so_depth_metric_sample': (C.c_int, [_P, _P, _I, _I, _I, _I, _P, _P]),
    'so_depth_metric_sums': (C.c_int, [_P, _P, _P, _P, _I, _I, _P, _P]),
    'so_field_query': (C.c_int, [_P, _P, C.POINTER(VolumeDesc), _P, _L, _P, _P, _P, _P]),
    'so_occ_classify': (C.c_int, [_P, _P, C.POINTER(VolumeDesc), _P, _P, _P, _I, _I, _I, _P, C.POINTER(OccGrid), _P, _I, _P, _P,
                                  _P]),
    'so_occ_hist': (C.c_int, [_P, _P, _P, _L, _I, _P, _P]),
    'so_reproj_workspace_floats': (_L, [C.POINTER(ReprojDesc)]),
    'so_reproj_forward': (C.c_int, [C.POINTER(ReprojDesc)] + [_P] * 12),
    'so_reproj_backward': (C.c_int, [C.POINTER(ReprojDesc)] + [_P] * 13),
    'so_reproj_check_layout': (C.c_int, [_P, _L, _I, _P, _P]),
    'so_msda_forward': (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    'so_msda_backward': (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    'so_linear_force_ss': (C.c_int, [C.c_int]),
    'so_split_tf32': (C.c_int, [_P, _P, _P, _L, _P]),
    'so_linear_3xtf32': (C.c_int, [_P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _P]),
    'so_linear_3xtf32_ln': (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _F, _P, _L, _I, _I, _I, _P]),
    'so_flatten_level': (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _L, _L, _P]),
    'so_layer_norm': (C.c_int, [_P, _P, _P, _P, _P, _L, _I, _F, _P]),
    'so_point_sampling': (C.c_int, [_P, _P, _I, _I, _I, _F, _F, _P, _P, _P, _P]),
    'so_tpv_cross_attn_forward': (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    'so_tpv_cross_attn_forward_strided': (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P] + [_I] * 10 + [_P]),
    'so_tpv_self_attn_forward_strided': (C.c_int, [_P, _P, _P, _P, _P, _P, _P] + [_I] * 9 + [_P]),
    'so_attn_force_v1': (C.c_int, [C.c_int]),
    'so_visible_index_lists': (C.c_int, [_P, _I, _I, _I, _P, _P, _P]),
    'so_tpv_self_attn_forward': (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
}

_lib = None


class SelfOccLibraryError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and bind every declared symbol.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SelfOccLibraryError(
            'libselfocc_b200.so not found at %s -- run `python -c "import __graft_entry__ as g; g.build()"` '
            '(there is no CPU/PyTorch fallback for the hot path)' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise SelfOccLibraryError('symbol %s missing from %s' % (name, LIB_PATH)) from e
        fn.restype = res
        fn.argtypes = args
    if lib.so_abi_version() != ABI_VERSION:
        raise SelfOccLibraryError('ABI version mismatch: library %d, binding %d' % (lib.so_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(code, what):
    if code != 0:
        lib = load()
        raise SelfOccLibraryError('%s failed: %s (code %d, cudaError %d)' % (
            what, lib.so_error_string(code).decode(), code, lib.so_last_cuda_error()))


def launch_count():
    return int(load().so_launch_count())


PROF_TAGS = ('render_infer', 'tpv_decode', 'tpv_cross_attn', 'tpv_self_attn', 'msda_forward', 'msda_backward',
             'render_train_fwd', 'render_train_bwd', 'linear_3xtf32', 'reserved')


def profile_enable(on=True):
    load().so_profile_enable(int(on))
    load().so_profile_reset()


def profile_reset():
    load().so_profile_reset()


def profile_read():
    """{tag: (total_ms, calls)} since the last reset; the stream must be synchronised first."""
    lib = load()
    out = {}
    for i, t in enumerate(PROF_TAGS):
        ms, n = C.c_float(0), C.c_int32(0)
        check(lib.so_profile_elapsed_ms(i, C.byref(ms), C.byref(n)), 'so_profile_elapsed_ms')
        if n.value:
            out[t] = (ms.value, n.value)
    return out
