"""ctypes binding of libunetsulc_b200.so (the C-ABI declared in include/unetsulc_b200.h).

The library is the product path.  There is no fallback: if it cannot be loaded, every op raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libunetsulc_b200.so")

_vp, _i, _ll, _f = C.c_void_p, C.c_int, C.c_longlong, C.c_float

# name -> (restype, argtypes); must list every symbol include/unetsulc_b200.h declares
SIGNATURES = {
    "b2_last_error": (C.c_char_p, []),
    "b2_conv3d_igemm": (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "b2_conv3d_splitk_workspace_bytes": (_ll, [_i, _i, _i, _i, _i]),
    "b2_conv3d_igemm_splitk": (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _ll, _vp]),
    "b2_conv3d_igemm_stats": (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "b2_conv3d_igemm_bstats": (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "b2_relu_gn_finalize_acc": (_i, [_vp, _ll, _i, _i, _f, _vp, _vp, _vp, _vp, _vp]),
    "b2_relu_gn_bwd_acc": (_i, [_vp, _vp, _i, _i, _vp, _ll, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp]),
    "b2_conv3d_igemm_bias": (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _ll,
                                  _vp]),
    "b2_conv3d_first_fwd_bias": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "b2_relu_gn_bwd_dbias": (_i, [_vp, _i, _i, _vp, _i, _ll, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp, _vp,
                                  _vp]),
    "b2_relu_gn_bwd_acc_dbias": (_i, [_vp, _vp, _i, _i, _vp, _ll, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp,
                                      _vp, _vp]),
    "b2_conv3d_wgrad_workspace_bytes": (_ll, [_i, _i, _i, _i, _i, _i]),
    "b2_conv3d_wgrad": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp]),
    "b2_conv3d_wgrad_partial": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "b2_wgrad_reduce_multi": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "b2_conv3d_first_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "b2_conv3d_first_fwd_stats": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "b2_conv3d_first_wgrad_workspace_bytes": (_ll, [_i]),
    "b2_conv3d_first_wgrad": (_i, [_vp, _vp, _i, _i, _vp, _vp, _ll, _i, _i, _i, _i, _i, _vp]),
    "b2_gn_workspace_bytes": (_ll, [_i, _i]),
    "b2_relu_gn_stats": (_i, [_vp, _i, _ll, _i, _i, _f, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp]),
    "b2_relu_gn_apply": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "b2_relu_gn_bwd_workspace_bytes": (_ll, [_i, _i]),
    "b2_relu_gn_bwd": (_i, [_vp, _i, _i, _vp, _i, _ll, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp]),
    "b2_maxpool3d_bwd_add": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b2_maxpool3d_bwd_add_bstats": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "b2_upcat_fwd": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    "b2_upcat_bwd": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp]),
    "b2_upcat_bwd_workspace_bytes": (_ll, [_i, _i, _i, _i, _i]),
    "b2_upcat_bwd_separable": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _ll, _vp]),
    "b2_upcat_bwd_separable_bstats": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _ll, _vp, _vp, _vp]),
    "b2_head_workspace_bytes": (_ll, [_i]),
    "b2_head_ce": (_i, [_vp, _vp, _ll, _vp, _vp, _i, _i, _f, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp,
                        _vp]),
    "b2_head_ce_bstats": (_i, [_vp, _vp, _ll, _vp, _vp, _i, _i, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp,
                               _vp, _vp, _i, _vp]),
    "b2_head_gather": (_i, [_vp, _vp, _ll, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "b2_head_dense_fwd": (_i, [_vp, _i, _ll, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "b2_head_dense_bwd": (_i, [_vp, _vp, _i, _ll, _vp, _i, _i, _vp, _vp, _vp, _vp, _ll, _vp]),
    "b2_sgd_step": (_i, [_vp, _vp, _vp, _vp, _i, _f, _f, _f, _vp]),
    "b2_pack_conv_weights": (_i, [_vp, _vp, _vp, _i, _i, _vp]),
    "b2_pack_conv_weights_multi": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "b2_scatter_volume_workspace_bytes": (_ll, [_i, _i, _i]),
    "b2_scatter_volume": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _ll, _vp, _ll, _vp]),
    "b2_scatter_volume_rot_workspace_bytes": (_ll, [_i, _i, _i, _i]),
    "b2_scatter_volume_rot": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _vp, _vp, _ll, _vp, _vp, _ll, _vp]),
    "b2_fold_vote_workspace_bytes": (_ll, [_ll, _i, _i, _i]),
    "b2_fold_vote": (_i, [_vp, _vp, _ll, _i, _i, _vp, _i, _vp, _vp, _ll, _vp]),
    "b2_match_voxels_workspace_bytes": (_ll, [_i]),
    "b2_match_voxels": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _ll, _vp]),
    "b2_esi_counts": (_i, [_vp, _vp, _ll, _i, _vp, _vp]),
    "b2_exact_split3": (_i, [_vp, _ll, _i, _i, _i, _vp, _vp]),
    "b2_exact_split_first": (_i, [_vp, _ll, _vp, _vp]),
    "b2_exact_gn_workspace_bytes": (_ll, [_i]),
    "b2_exact_gn_stats": (_i, [_vp, _ll, _i, _i, _f, _vp, _vp, _vp, _vp, _ll, _vp]),
    "b2_exact_gn_apply": (_i, [_vp, _ll, _i, _vp, _vp, _i, _i, _vp]),
    "b2_exact_maxpool": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "b2_exact_upsample": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    "b2_exact_head_gather": (_i, [_vp, _vp, _ll, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "b2_step_metrics": (_i, [_vp, _vp, _ll, _i, _vp, _vp, C.c_double, _vp, _vp]),
}

_lib = None


def load():
    """Loads the shared library (once).  Raises RuntimeError when it is missing — never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libunetsulc_b200.so not built (%s). Run __graft_entry__.build() or "
            "python 2022_pauriau_unetsulc_b200/build.py; there is no CPU/PyTorch fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, name):
    if rc != 0:
        msg = load().b2_last_error()
        raise RuntimeError("%s failed (%d): %s" % (name, rc, msg.decode() if msg else "?"))
