"""ctypes binding of libdiffnet_fem.so (C ABI: include/diffnet_fem.h).

The library is the product; this file only marshals pointers, sizes and strides.  There is no
CPU fallback: if the shared object is missing the import of any op raises with build
instructions, and every entry point refuses non-sm_100 devices (DN_EARCH).
"""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DIFFNET_FEM_LIB", os.path.join(PKG, "lib", "libdiffnet_fem.so"))

DN_MAX_MASKS = 3
DN_OK, DN_EINVAL, DN_EARCH, DN_ECUDA, DN_EWORKSPACE, DN_ENOSTREAM = 0, -1, -2, -3, -4, -5
DN_F_LOAD_VECTOR = 1


class dn_field(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("stride_b", C.c_int64), ("stride_z", C.c_int64),
                ("stride_y", C.c_int64)]


class dn_mask(C.Structure):
    _fields_ = [("mask", dn_field), ("value_field", dn_field), ("value", C.c_float),
                ("_pad", C.c_int32)]


class dn_geom(C.Structure):
    _fields_ = [("nsd", C.c_int32), ("batch", C.c_int32), ("nx", C.c_int32), ("ny", C.c_int32),
                ("nz", C.c_int32), ("ngp_1d", C.c_int32), ("hx", C.c_double), ("hy", C.c_double),
                ("hz", C.c_double), ("z_own_lo", C.c_int32), ("z_own_hi", C.c_int32),
                ("mean_count", C.c_double)]


class dn_consts(C.Structure):
    _fields_ = [("c_k", C.c_double), ("c_f", C.c_double), ("scale", C.c_double),
                ("reduction", C.c_int32), ("flags", C.c_int32)]


class dn_slab_link(C.Structure):
    _fields_ = [("halo_plane", C.c_void_p * 2), ("halo_flag", C.c_void_p * 2), ("put_dst", C.c_void_p * 2),
                ("put_flag", C.c_void_p * 2), ("put_plane", C.c_int32 * 2), ("loss_slots", C.c_void_p),
                ("step", C.c_void_p), ("tickets", C.c_void_p), ("status", C.c_void_p),
                ("max_spins", C.c_int64), ("rank", C.c_int32), ("world", C.c_int32)]


_P = C.POINTER
_ENERGY_ARGS = [_P(dn_field), _P(dn_field), _P(dn_field), _P(dn_field), _P(dn_mask), C.c_int,
                _P(dn_field), _P(dn_geom), _P(dn_consts), C.c_void_p, C.c_void_p, C.c_void_p,
                C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
_RESID_ARGS = [_P(dn_field), _P(dn_field), _P(dn_field), _P(dn_mask), C.c_int, C.c_int, _P(dn_geom),
               C.c_double, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
_GP_ARGS = [_P(dn_field), _P(dn_geom), C.c_int, C.c_void_p, C.c_void_p]
_GPADJ_ARGS = [C.c_void_p, _P(dn_geom), C.c_int, C.c_void_p, C.c_void_p]
_GPM_ARGS = [_P(dn_field), _P(dn_geom), C.c_int, _P(C.c_int), _P(C.c_void_p), C.c_void_p]
_EIG_ARGS = [_P(dn_field), _P(dn_field), _P(dn_field), _P(dn_field), _P(dn_mask), C.c_int, _P(dn_field),
             _P(dn_geom), _P(dn_consts), C.c_void_p, C.c_void_p, _P(C.c_void_p), C.c_void_p]
_RIG_ARGS = [_P(dn_field), _P(dn_field), _P(dn_field), _P(dn_field), _P(dn_mask), C.c_int, _P(dn_geom), C.c_double,
             C.c_void_p, C.c_void_p, _P(C.c_void_p), C.c_void_p]
_GPMADJ_ARGS = [_P(C.c_void_p), _P(dn_geom), C.c_int, _P(C.c_int), C.c_void_p, C.c_void_p]

# symbol -> (restype, argtypes); tests/test_abi.py checks this table against include/diffnet_fem.h
PROTOTYPES = {
    "dn_abi_version": (C.c_int, []),
    "dn_last_error": (C.c_char_p, []),
    "dn_device_check": (C.c_int, []),
    "dn_fem_workspace_bytes": (C.c_size_t, [_P(dn_geom)]),
    "dn_debug_plan": (C.c_int, [_P(dn_geom), C.c_int, C.c_int, C.POINTER(C.c_int64)]),
    "dn_fem_energy_2d_f32": (C.c_int, _ENERGY_ARGS),
    "dn_fem_energy_3d_f32": (C.c_int, _ENERGY_ARGS),
    "dn_fem_energy_3d_linked_f32": (C.c_int, [_P(dn_field), _P(dn_field), _P(dn_field), _P(dn_mask), C.c_int,
                                              _P(dn_field), _P(dn_geom), _P(dn_consts), _P(dn_slab_link),
                                              C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                              C.c_void_p]),
    "dn_peer_loss_sum_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "dn_fem_residual_2d_f32": (C.c_int, _RESID_ARGS),
    "dn_fem_residual_3d_f32": (C.c_int, _RESID_ARGS),
    "dn_fem_energy_input_grads_2d_f32": (C.c_int, _EIG_ARGS),
    "dn_fem_energy_input_grads_3d_f32": (C.c_int, _EIG_ARGS),
    "dn_fem_residual_input_grads_2d_f32": (C.c_int, _RIG_ARGS),
    "dn_fem_residual_input_grads_3d_f32": (C.c_int, _RIG_ARGS),
    "dn_fem_gp_eval_2d_f32": (C.c_int, _GP_ARGS),
    "dn_fem_gp_eval_3d_f32": (C.c_int, _GP_ARGS),
    "dn_fem_gp_eval_adj_2d_f32": (C.c_int, _GPADJ_ARGS),
    "dn_fem_gp_eval_adj_3d_f32": (C.c_int, _GPADJ_ARGS),
    "dn_fem_gp_eval_multi_2d_f32": (C.c_int, _GPM_ARGS),
    "dn_fem_gp_eval_multi_3d_f32": (C.c_int, _GPM_ARGS),
    "dn_fem_gp_eval_multi_adj_2d_f32": (C.c_int, _GPMADJ_ARGS),
    "dn_fem_gp_eval_multi_adj_3d_f32": (C.c_int, _GPMADJ_ARGS),
    "dn_fem_gp_eval_general_f32": (C.c_int, [_P(dn_field), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                             _P(C.c_float), C.c_void_p, C.c_void_p]),
    "dn_fem_gp_eval_general_adj_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                 _P(C.c_float), C.c_void_p, C.c_void_p]),
    "dn_fem_load_vector_f32": (C.c_int, [_P(dn_field), _P(dn_geom), C.c_void_p, C.c_void_p]),
    "dn_gen_kl_table_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "dn_gen_kl_inputs_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _P(C.c_double), C.c_double, C.c_int, C.c_int,
                                       C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dn_gen_image_inputs_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dn_gen_voxel_inputs_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "dn_gen_star_inputs_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dn_gen_box_masks_3d_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dn_scale_inplace_f32": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "dn_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "dn_peer_free": (C.c_int, [C.c_void_p]),
    "dn_peer_export": (C.c_int, [C.c_void_p, C.c_char_p]),
    "dn_peer_import": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "dn_peer_unimport": (C.c_int, [C.c_void_p]),
    "dn_peer_put_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dn_peer_allreduce_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                        C.c_int64, C.c_void_p, C.c_void_p]),
    "dn_peer_wait_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int64,
                                   C.c_void_p, C.c_void_p]),
}

_lib = None


class DiffNetFEMError(RuntimeError):
    code = None        # the dn_status the library returned, when the error came from a call


def lib():
    """Load (once) and return the shared library; fail loudly if it was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DiffNetFEMError(
                f"{LIB_PATH} not found. diffnet_b200 has no CPU or PyTorch fallback: build the "
                "sm_100a library first with `python -m diffnet_b200.build` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`).")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)      # AttributeError = ABI mismatch, also loud
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc: int, what: str):
    if rc != DN_OK:
        msg = lib().dn_last_error()
        err = DiffNetFEMError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
        err.code = rc
        raise err
