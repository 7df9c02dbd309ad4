"""ctypes binding of the C-ABI library (include/fastpcc_b200.h).

There is no CPU fallback: if libfastpcc_b200.so is missing or does not load, importing the product path
fails loudly.  `build.build()` compiles it in-tree with nvcc for sm_100a.
"""
import ctypes as C
import os.path as osp

from . import build as _build

_vp, _i, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t


class Epilogue(C.Structure):
    """fpcc_epilogue (include/fastpcc_b200.h)"""
    _fields_ = [('bias', _vp), ('slope', _vp), ('requant_mul', _vp), ('zero_point', _vp),
                ('shift', C.c_int32), ('out_type', C.c_int32), ('mul_is_scalar', C.c_int32),
                ('residual', _vp), ('post_slope', _vp), ('row_bias', _vp), ('row_idx', _vp), ('row_bias_bound', C.c_int32),
                ('post_requant_mul', _vp), ('post_zero_point', _vp), ('post_shift', C.c_int32), ('post_requant_slope', _vp), ('aux_out', _vp), ('out_ld', C.c_int64)]


_EP = C.POINTER(Epilogue)

# name -> (restype, argtypes); every symbol declared in include/fastpcc_b200.h
SIGNATURES = {
    'fpcc_last_error': (C.c_char_p, []),
    'fpcc_version': (_i, []),
    'fpcc_device_check': (_i, [_vp, _vp, _vp]),
    'fpcc_hash_insert_coords': (_i, [_vp, _vp, _i, _vp, _i, _i, _vp]),
    'fpcc_kmap_lookup': (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _i64, _vp]),
    'fpcc_kmap_compact_workspace': (_sz, [_i, _i]),
    'fpcc_kmap_compact': (_i, [_vp, _i, _i, _i64, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    'fpcc_kmap_from_parent': (_i, [_vp, _i64, _i, _vp, _vp, _vp, _vp, _i, _vp, _i64, _vp]),
    'fpcc_kmap_row_masks': (_i, [_vp, _i, _i, _i64, _vp, _vp]),
    'fpcc_kmap_permute': (_i, [_vp, _i, _i, _i64, _vp, _vp, _i64, _vp]),
    'fpcc_scan_workspace': (_sz, [_i]),
    'fpcc_downsample': (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'fpcc_upsample': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'fpcc_occ_to_bits': (_i, [_vp, _i, _vp, _vp]),
    'fpcc_gather_patches': (_i, [_vp, _i, _vp, _i64, _i, _i, _vp, _i, _vp]),
    'fpcc_occ_bits_q8': (_i, [_vp, _i64, _i, _i, _vp, _i64, _vp]),
    'fpcc_slot_table': (_i, [_vp, _vp, _i, _vp, _i64, _vp]),
    'fpcc_morton_encode': (_i, [_vp, _i64, _i, _i, _vp, _vp]),
    'fpcc_gather_rows16': (_i, [_vp, _vp, _i64, _vp, _vp]),
    'fpcc_voxelize_workspace': (_sz, [_i64]),
    'fpcc_voxelize_f32': (_i, [_vp, _i64, _i, C.c_float, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    'fpcc_kd_split_workspace': (_sz, [_i64, _i]),
    'fpcc_kd_split': (_i, [_vp, _i64, _i, _vp, _vp, _vp, _sz, _vp]),
    'fpcc_frame_header_write': (_i, [_vp, _i, _vp]),
    'fpcc_frame_header_read': (_i, [_vp, _i64, _vp, _vp]),
    'fpcc_partitions_pack': (_i64, [_vp, _vp, _i, _vp, _i64]),
    'fpcc_partitions_index': (_i, [_vp, _i64, _i, _vp, _vp]),
    'fpcc_bytes_list_concat': (_i64, [_vp, _vp, _i, _vp, _i64]),
    'fpcc_bytes_list_split': (_i64, [_vp, _i64, _i, _vp, _vp]),
    'fpcc_nn_search': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    'fpcc_knn_workspace': (_sz, [_i64, _i]),
    'fpcc_knn_search': (_i, [_i, _i, _i, _vp, _i64, _i, _i, _i, _vp, _i64, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'fpcc_nn_tie_attr': (_i, [_i, _vp, _i64, _i, _i, _i, _vp, _i64, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'fpcc_knn_normals': (_i, [_i, _i, _vp, _i64, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'fpcc_gemm_i8': (_i, [_vp, _vp, _vp, _i, _vp, _i, _i, _i, _vp]),
    'fpcc_gather_gemm_scatter_i8': (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'fpcc_requant': (_i, [_vp, _i64, _i, _EP, _vp, _vp]),
    'fpcc_requant_ld': (_i, [_vp, _i64, _i, _EP, _vp, _i64, _vp]),
    'fpcc_prelu_i32': (_i, [_vp, _i64, _vp, _vp, _vp]),
    'fpcc_spconv_i8': (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _i64, _i, _vp, _vp, _EP, _vp, _vp]),
    'fpcc_linear_i8': (_i, [_vp, _i, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _EP, _vp, _vp]),
    'fpcc_spconv_f16': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _vp, _i64, _i, _vp, _vp, _i, C.c_float, _vp, _i, C.c_float, _vp, _i, _vp]),
    'fpcc_spconv_wgrad_f16': (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _i, _i, _vp]),
    'fpcc_kmap_transpose': (_i, [_vp, _i, _i, _i64, _i, _vp, _i64, _vp]),
    'fpcc_act_grad_workspace': (_sz, [_i64, _i]),
    'fpcc_act_grad_f16': (_i, [_vp, _i, _i64, _vp, _i, _i64, _i64, _i, _i, C.c_float, _vp, _i, _i, _vp, _vp, _sz, _vp]),
    'fpcc_linear_f16': (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _vp, _i, C.c_float, _vp, _i, C.c_float, _vp, _i, _vp]),
    'fpcc_set_tc_mode': (_i, [_i]),
    'fpcc_set_sm_budget': (_i, [_i]),
    'fpcc_set_blocking_sync': (_i, [_i]),
    'fpcc_mma_i8_peak': (_i, [_i, _i, _vp, _vp]),
    'fpcc_gemm_engine': (_i, [_i, _i, _i, _i]),
    'fpcc_softmax_i32': (_i, [_vp, _i64, _i, _vp, _vp]),
    'fpcc_quantize_cdf': (_i, [_vp, _i64, _i64, _i, _vp, _i, _vp]),
    'fpcc_cdf_symbol_ranges': (_i, [_vp, _i64, _i64, _i, _vp, _vp, _vp]),
    'fpcc_table_symbol_ranges': (_i, [_vp, _i64, _i, _vp, _i64, _vp, _vp]),
    'fpcc_rans_encode': (_i, [_vp, _vp, _vp, _i, _i64, _vp, _i64, _vp, _vp, _i, _vp, _sz, _vp]),
    'fpcc_rans_dec_init': (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    'fpcc_rans_decode': (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _vp, _i, _vp, _i, _vp, _vp]),
    'fpcc_rans_binary_ranges': (_i, [_vp, _vp, _i64, _vp, _vp]),
    'fpcc_rans_binary_decode': (_i, [_vp, _vp, _vp, _vp, _i64, _i, _vp, _vp, _vp]),
    'fpcc_indexed_count': (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _i64, _i, _vp, _vp]),
    'fpcc_indexed_ranges': (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    'fpcc_indexed_decode': (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _i64, _i, _vp, _vp, _vp]),
    'fpcc_pmf_to_quantized_cdf': (_i, [_vp, _i, _i, _vp, _i, _vp, _vp, _vp]),
    'fpcc_factorized_bits': (_i, [_vp, _i64, _i64, _i, _vp, C.c_float, _vp, _vp]),
    'fpcc_factorized_grad_workspace': (_sz, [_i64, _i]),
    'fpcc_factorized_grad': (_i, [_vp, _i64, _vp, _i64, _i64, _i, _vp, C.c_float, _vp, _vp, _vp, _sz, _vp]),
    'fpcc_factorized_pmf': (_i, [_vp, _i, _i, _i, _vp, _vp]),
    'fpcc_gaussian_bits': (_i, [_vp, _i64, _vp, _i64, _vp, _i64, _i64, _i, C.c_float, C.c_float, _vp, _vp]),
    'fpcc_gaussian_grad': (_i, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i, C.c_float, C.c_float, _vp, _vp, _vp, _vp]),
    'fpcc_gaussian_tail_multiplier': (C.c_double, [C.c_double]),
    'fpcc_gaussian_pmf': (_i, [_vp, _i, C.c_double, _i, _vp, _vp, _vp]),
    'fpcc_gaussian_indexes': (_i, [_vp, _i64, _vp, _i64, _vp, _i64, _i64, _i, C.c_float, _vp, _i, _vp, _vp, _vp]),
}

_LIB = None


def so_path():
    # FPCC_LIB_PATH: an experiment build of the SAME library (build.build_variant) for A/B timing; there is still no
    # fallback of any kind: the named file must exist and export every declared symbol
    import os
    return os.environ.get('FPCC_LIB_PATH') or _build.SO


def load(build_if_missing=True):
    """Loads libfastpcc_b200.so; raises (never falls back) when it cannot."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = so_path()
    if not osp.isfile(path):
        if not build_if_missing:
            raise RuntimeError(f'{path} is missing: run `python -m fastpcc_b200.build` (nvcc, sm_100a)')
        _build.build()
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


def check(rc, what=''):
    if rc != 0:
        msg = load().fpcc_last_error()
        raise RuntimeError(f'{what}: {msg.decode() if msg else "error %d" % rc}')


def call(name, *args):
    check(getattr(load(), name)(*args), name)
