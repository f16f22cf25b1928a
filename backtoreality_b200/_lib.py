"""ctypes binding of libb2r.so (the C ABI declared in include/b2r.h).

There is NO fallback: if the library is missing or a call fails this module raises.  The
library is built in-tree by `backtoreality_b200.build.build()` (nvcc, sm_100a only).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B2R_LIB: another build of the same C ABI (A/B timing of kernel variants); default: the in-tree build
LIB_PATH = os.environ.get("B2R_LIB") or os.path.join(_HERE, "libb2r.so")

_vp = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float
_ip = ctypes.POINTER(ctypes.c_int)

# name -> argtypes; every function returns int (b2r_status) unless listed in _RESTYPES
SIGNATURES = {
    "b2r_version": [],
    "b2r_status_string": [_i],
    "b2r_last_error": [],
    "b2r_struct_bytes": [_i],
    "b2r_ref_block_threads": [_i],
    "b2r_fps": [_vp, _i, _i, _i, _vp, _vp],
    "b2r_fps_ex": [_vp, _i, _i, _i, _vp, _i, _vp],
    "b2r_fps_plan": [_i, _i, _ip, _ip, _ip, _ip],
    "b2r_fps_workspace_bytes": [_i, _i],
    "b2r_fps_ws": [_vp, _i, _i, _i, _vp, _i, _vp, ctypes.c_longlong, _vp],
    "b2r_fps_sort": [_vp, _i, _i, _vp, ctypes.c_longlong, _vp],
    "b2r_fps_ws_presorted": [_vp, _i, _i, _i, _vp, _i, _vp, ctypes.c_longlong, _vp],
    "b2r_gather_fwd": [_vp, _vp, _i, _i, _i, _i, _vp, _vp],
    "b2r_gather_bwd": [_vp, _vp, _i, _i, _i, _i, _vp, _vp],
    "b2r_ball_query": [_vp, _vp, _i, _i, _i, _f, _i, _vp, _vp],
    "b2r_ball_query_workspace_bytes": [_i, _i],
    "b2r_ball_query_grid": [_vp, _vp, _i, _i, _i, _f, _i, _vp, _vp, ctypes.c_longlong, _vp],
    "b2r_group_fwd": [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp],
    "b2r_group_bwd": [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp],
    "b2r_three_nn": [_vp, _vp, _i, _i, _i, _vp, _vp, _vp],
    "b2r_three_interp_fwd": [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp],
    "b2r_three_interp_bwd": [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp],
    "b2r_scatter_plan_bytes": [_i, ctypes.c_longlong, _i, _i, _i],
    "b2r_scatter_plan": [_vp, _vp, _i, ctypes.c_longlong, _i, _i, _vp, ctypes.c_longlong, _vp],
    "b2r_group_bwd_plan": [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp],
    "b2r_three_interp_bwd_plan": [_vp, _vp, _i, _i, _i, _i, _vp, _vp],
    "b2r_adam_state_bytes": [],
    "b2r_adam_flat_step": [_vp, _vp, _vp, _vp, ctypes.c_longlong, _vp, _f, _f, _f, _f, _f, _f, _vp],
    "b2r_nn_argmin": [_vp, _vp, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp],
    "b2r_query_group_fwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _vp, _vp],
    "b2r_query_group_bwd": [_vp, _vp, _i, _i, _i, _i, _i, _f, _i, _vp, _vp, _vp, _vp],
}
_RESTYPES = {"b2r_status_string": ctypes.c_char_p, "b2r_last_error": ctypes.c_char_p,
             "b2r_fps_workspace_bytes": ctypes.c_longlong,
             "b2r_scatter_plan_bytes": ctypes.c_longlong,
             "b2r_ball_query_workspace_bytes": ctypes.c_longlong,
             "b2r_mlp_weight_image_bytes": ctypes.c_longlong}


class SaLayer(ctypes.Structure):
    """struct b2r_sa_layer (include/b2r.h)."""
    _fields_ = [
        ("B", _i), ("N", _i), ("NP", _i), ("NS", _i), ("Cin", _i), ("Cout", _i),
        ("mode", _i), ("epilogue", _i),
        ("xyz", _vp), ("new_xyz", _vp), ("feat_t", _vp), ("idx", _vp),
        ("radius", _f), ("normalize_xyz", _i),
        ("z_prev", _vp), ("scale_prev", _vp), ("shift_prev", _vp),
        ("w_image", _vp), ("z", _vp), ("stats", _vp),
        ("zmax", _vp), ("zmin", _vp), ("amax", _vp), ("amin", _vp),
        ("sm_limit", _i),
        ("cidx", _vp), ("ccen", _vp), ("cmeta", _vp),
        ("co0", _i), ("co_n", _i), ("ci0", _i), ("ci_n", _i), ("accumulate", _i),
    ]


_ip = ctypes.POINTER(_i)
SIGNATURES.update({
    "b2r_mlp_weight_image_bytes": [_i, _i, _i],
    "b2r_mlp_pack_weight": [_vp, _i, _i, _i, _vp, _vp],
    "b2r_sa_layer_fwd": [ctypes.POINTER(SaLayer), _vp],
    "b2r_sa_layer_fwd_supported": [_i, _i, _i, _i, _i, _i, _i],
    "b2r_sa_layer_fwd_slices": [_i, _i, _i, _i, _ip, _ip],
    "b2r_bn_finalize": [_vp, _i, ctypes.c_double, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp,
                        _vp, _vp],
    "b2r_bn_finalize_dev": [_vp, _i, ctypes.c_double, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp,
                            _vp, _vp, _vp],
    "b2r_pool_finalize": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp],
    "b2r_to_point_major": [_vp, _i, _i, _i, _vp, _vp],
})



class SaLayerBwd(ctypes.Structure):
    """struct b2r_sa_layer_bwd_desc (include/b2r.h)."""
    _fields_ = [
        ("B", _i), ("N", _i), ("NP", _i), ("NS", _i), ("Cin", _i), ("Cout", _i), ("mode", _i),
        ("xyz", _vp), ("new_xyz", _vp), ("feat_t", _vp), ("idx", _vp),
        ("radius", _f), ("normalize_xyz", _i),
        ("z_prev", _vp), ("scale_prev", _vp), ("shift_prev", _vp),
        ("w_image_bf16", _vp), ("dz", _vp), ("gr", _vp), ("z", _vp),
        ("dysel", _vp), ("asel", _vp),
        ("coef_a", _vp), ("coef_b", _vp), ("coef_c", _vp),
        ("dW", _vp), ("gr_prev", _vp), ("stats_prev", _vp),
        ("g_feat_t", _vp), ("g_xyz", _vp), ("g_new_xyz", _vp),
        ("sm_limit", _i),
        ("cidx", _vp), ("ccen", _vp), ("cmeta", _vp),
        ("co0", _i), ("co_n", _i), ("ci0", _i), ("ci_n", _i), ("accumulate", _i),
    ]


SIGNATURES.update({
    "b2r_mlp_weight_bf16_image_bytes": [_i, _i, _i],
    "b2r_mlp_pack_weight_bf16": [_vp, _i, _i, _i, _vp, _vp],
    "b2r_sa_layer_bwd": [ctypes.POINTER(SaLayerBwd), _vp],
    "b2r_sa_layer_bwd_supported": [_i, _i, _i, _i, _i, _i, _i],
    "b2r_sa_layer_bwd_slices": [_i, _i, _i, _i, _ip, _ip],
    "b2r_pool_bwd_prep": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp],
    "b2r_bn_bwd_finalize": [_vp, _i, ctypes.c_double, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp,
                            _vp, _vp, _vp, _vp],
})
_RESTYPES["b2r_mlp_weight_bf16_image_bytes"] = ctypes.c_longlong

# pad-free position space of a fused SA block (csrc/compact.cu)
SIGNATURES.update({
    "b2r_compact_capacity": [_i, _i, _i],
    "b2r_compact_workspace_bytes": [_i, _i],
    "b2r_compact_plan": [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "b2r_sa_layer_fwd_tile": [_i] * 8,
    "b2r_sa_layer_bwd_tile": [_i] * 9,
})
_RESTYPES["b2r_compact_capacity"] = ctypes.c_longlong
_RESTYPES["b2r_compact_workspace_bytes"] = ctypes.c_longlong



class DenseLayer(ctypes.Structure):
    """struct b2r_dense_layer (include/b2r.h)."""
    _fields_ = [
        ("M", _i), ("Cin", _i), ("Cout", _i),
        ("in_", _vp), ("ld_in", _i), ("sc_in", _vp), ("sh_in", _vp),
        ("w_img", _vp), ("bias", _vp), ("z", _vp), ("ld_z", _i), ("stats", _vp),
    ]


class DenseLayerBwd(ctypes.Structure):
    """struct b2r_dense_layer_bwd (include/b2r.h)."""
    _fields_ = [
        ("M", _i), ("Cin", _i), ("Cout", _i),
        ("in_", _vp), ("ld_in", _i), ("sc_in", _vp), ("sh_in", _vp),
        ("g", _vp), ("zz", _vp), ("ld_g", _i),
        ("ca", _vp), ("cb", _vp), ("cc", _vp),
        ("wt_img", _vp), ("gin", _vp), ("ld_gin", _i), ("stats_in", _vp), ("dW", _vp),
    ]


_ll = ctypes.c_longlong
SIGNATURES.update({
    "b2r_bn_bwd_finalize_ex": [_vp, _i, ctypes.c_double, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp,
                               _vp, _vp, _vp, _vp, _vp],
    "b2r_dense_image_bytes": [_i, _i],
    "b2r_dense_pack": [_vp, _i, _i, _vp, _vp, _vp],
    "b2r_dense_fwd": [ctypes.POINTER(DenseLayer), _vp],
    "b2r_dense_bwd": [ctypes.POINTER(DenseLayerBwd), _vp],
    "b2r_interp_cat_fwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp],
    "b2r_interp_cat_bwd": [_vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "b2r_vote_tail_fwd": [_vp, _i, _vp, _vp, _ll, _i, _vp, _vp, _vp, _vp],
    "b2r_vote_tail_bwd": [_vp, _vp, _vp, _vp, _ll, _i, _i, _vp, _vp, _vp],
})
_RESTYPES["b2r_dense_image_bytes"] = ctypes.c_longlong


ADAM_MAX_GROUPS = 64    # B2R_ADAM_MAX_GROUPS


class AdamGroup(ctypes.Structure):
    """struct b2r_adam_group (include/b2r.h): one entry of the device table."""
    _fields_ = [("start", _ll), ("end", _ll), ("lr", _f), ("weight_decay", _f)]


class AdamDesc(ctypes.Structure):
    """struct b2r_adam_desc (include/b2r.h)."""
    _fields_ = [
        ("params", _vp), ("grads", _vp), ("exp_avg", _vp), ("exp_avg_sq", _vp), ("n", _ll),
        ("state", _vp), ("groups", _vp), ("n_groups", _i),
        ("beta1", _f), ("beta2", _f), ("eps", _f), ("grad_scale", _f), ("decoupled", _i),
        ("clip_coef", _vp),
    ]


SIGNATURES.update({
    "b2r_adam_flat_step_groups": [ctypes.POINTER(AdamDesc), _vp],
    "b2r_flat_grad_norm_workspace_bytes": [_ll],
    "b2r_flat_grad_norm": [_vp, _ll, _f, _f, _vp, _vp, _vp, _vp],
})
_RESTYPES["b2r_flat_grad_norm_workspace_bytes"] = ctypes.c_longlong

_lib = None


class B2RError(RuntimeError):
    """A libb2r call returned a negative status."""


def lib():
    """Load libb2r.so once.  Raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError(
                "libb2r.so not found at %s -- build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or PyTorch fallback for these ops)" % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(l, name)  # AttributeError if the .so is stale: loud on purpose
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, ctypes.c_int)
        _lib = l
    return _lib


def check(status, what):
    if status != 0:
        l = lib()
        raise B2RError("%s failed: %s (%s)" % (
            what, l.b2r_status_string(status).decode(), l.b2r_last_error().decode()))
