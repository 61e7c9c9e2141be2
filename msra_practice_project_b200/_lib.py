"""ctypes binding of ``include/b2r.h`` (libb2r.so, sm_100a).

The library is the product; there is no fallback.  ``lib()`` raises ``RuntimeError`` when the
shared object is missing (run ``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C
msra_practice_project_b200/csrc``), and every call raises ``RuntimeError`` with
``b2r_last_error()`` on a non-zero return code.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb2r.so")

c_float_p = C.c_void_p      # device pointers travel as integers
c_ll = C.c_longlong


class MlpInput(C.Structure):
    """struct b2r_mlp_input (include/b2r.h)."""
    _fields_ = [("rays", C.c_void_p), ("z", C.c_void_p), ("x", C.c_void_p), ("n_rays", c_ll),
                ("n_samples", C.c_int), ("grid_n", C.c_int), ("grid_begin", c_ll), ("lattice_dims", C.c_int * 3),
                ("lattice_origin", C.c_float * 3), ("lattice_voxel", C.c_float)]


class LastSample(C.Structure):
    """struct b2r_last_sample (include/b2r.h)."""
    _fields_ = [("samples_per_ray", C.c_int), ("capacity", C.c_int), ("count", C.c_void_p), ("ray_ids", C.c_void_p),
                ("rel", C.c_float), ("abs", C.c_float)]


# name -> (restype, argtypes); must list every symbol include/b2r.h declares (checked by tests/test_abi.py)
SIGNATURES = {
    "b2r_last_error": (C.c_char_p, []),
    "b2r_version": (C.c_int, []),
    "b2r_device_ok": (C.c_int, []),
    "b2r_raygen": (C.c_int, [C.POINTER(C.c_double), C.c_int, C.c_int, C.c_double, C.c_int, c_ll, c_ll, c_float_p, C.c_void_p]),
    "b2r_raygen_poses": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, c_float_p, C.c_void_p]),
    "b2r_stratified_z": (C.c_int, [c_float_p, c_float_p, c_ll, C.c_int, c_float_p, c_float_p, C.c_void_p]),
    "b2r_composite_fwd": (C.c_int, [c_float_p, c_float_p, c_float_p, C.c_int, c_ll, C.c_int, c_float_p, c_float_p,
                                    c_float_p, c_float_p, C.c_void_p]),
    "b2r_composite_fwd_strided": (C.c_int, [c_float_p, c_float_p, c_float_p, C.c_int, c_ll, C.c_int, c_float_p, C.c_int, c_float_p, C.c_int,
                                            c_float_p, C.c_int, c_float_p, C.c_void_p]),
    "b2r_composite_bwd": (C.c_int, [c_float_p, c_float_p, c_float_p, C.c_int, c_ll, C.c_int, c_float_p, c_float_p,
                                    c_float_p, c_float_p, C.c_void_p]),
    "b2r_composite_loss_bwd": (C.c_int, [c_float_p, c_float_p, c_float_p, C.c_int, c_ll, C.c_int, c_float_p, c_float_p, c_float_p, c_float_p,
                                         C.c_float, c_float_p, c_float_p, C.c_void_p]),
    "b2r_train_loss_finish": (C.c_int, [c_float_p, c_float_p, C.c_float, c_float_p, c_float_p, c_float_p, C.c_void_p]),
    "b2r_sample_pdf": (C.c_int, [c_float_p, c_ll, c_float_p, c_ll, c_float_p, c_ll, C.c_int, C.c_int, c_float_p, C.c_int,
                                 c_float_p, c_float_p, c_float_p, C.c_void_p]),
    "b2r_sample_pdf_generic": (C.c_int, [c_float_p, c_ll, c_float_p, c_ll, c_float_p, c_ll, C.c_int, C.c_int, c_float_p, C.c_int,
                                 c_float_p, c_float_p, c_float_p, C.c_void_p]),
    "b2r_mlp_f32_workspace_bytes": (C.c_size_t, [C.c_int, c_ll, C.c_int]),
    "b2r_mlp_f32_fwd": (C.c_int, [C.c_int, c_float_p, c_float_p, C.c_int, C.POINTER(MlpInput), c_float_p, C.c_void_p,
                                  C.c_size_t, C.c_int, C.c_int, C.c_void_p]),
    "b2r_mlp_f32_bwd_scratch_bytes": (C.c_size_t, [C.c_int, c_ll]),
    "b2r_mlp_f32_bwd": (C.c_int, [C.c_int, c_float_p, c_float_p, C.c_int, C.POINTER(MlpInput), c_float_p, c_float_p,
                                  C.c_void_p, C.c_void_p, C.c_size_t, c_float_p, c_float_p, C.c_int, C.c_void_p]),
    "b2r_mlp_tc_packed_bytes": (C.c_size_t, [C.c_int]),
    "b2r_mlp_tc_pack": (C.c_int, [C.c_int, c_float_p, c_float_p, C.c_int, C.c_void_p, C.c_void_p]),
    "b2r_mlp_tc_fwd": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.POINTER(MlpInput), c_float_p, C.c_int, C.POINTER(LastSample), C.c_void_p]),
    "b2r_mlp_f32_last_sigma": (C.c_int, [C.c_int, c_float_p, c_float_p, C.c_int, C.c_int, c_ll, C.POINTER(MlpInput), C.c_int, C.c_void_p, C.c_int,
                                         c_float_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b2r_mlp_tc_train_saved_bytes": (C.c_size_t, [C.c_int, c_ll]),
    "b2r_mlp_tc_train_fwd": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(MlpInput), c_float_p, C.c_void_p, C.c_size_t, C.POINTER(LastSample), C.c_void_p]),
    "b2r_mlp_tc_bwd_packed_bytes": (C.c_size_t, [C.c_int]),
    "b2r_mlp_tc_pack_bwd": (C.c_int, [C.c_int, c_float_p, C.c_void_p, C.c_void_p]),
    "b2r_mlp_tc_train_scratch_bytes": (C.c_size_t, [C.c_int, c_ll]),
    "b2r_mlp_tc_pack_film_batched": (C.c_int, [c_float_p, c_float_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "b2r_mlp_tc_fwd_film_batched": (C.c_int, [C.c_void_p, C.c_int, c_ll, C.POINTER(MlpInput), c_float_p, C.c_int, C.POINTER(LastSample), C.c_void_p]),
    "b2r_to8b": (C.c_int, [c_float_p, c_ll, C.c_void_p, C.c_void_p]),
    "b2r_adam_step": (C.c_int, [c_float_p, c_float_p, c_float_p, c_float_p, c_ll, c_float_p, C.c_float, C.c_float, C.c_float, C.c_float,
                                C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "b2r_adam_step_floor": (C.c_int, [c_float_p, c_float_p, c_float_p, c_float_p, c_ll, c_float_p, C.c_float, C.c_float, C.c_float, C.c_float,
                                      C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "b2r_mlp_tc_train_bwd": (C.c_int, [C.c_int, C.c_void_p, c_ll, c_float_p, c_float_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                       c_float_p, C.c_void_p]),
    "b2r_mlp_tc_train_fwd_film_batched": (C.c_int, [C.c_void_p, C.c_int, c_ll, C.POINTER(MlpInput), c_float_p, C.c_void_p, C.c_size_t,
                                                    C.POINTER(LastSample), C.c_void_p]),
    "b2r_mlp_tc_pack_bwd_film": (C.c_int, [c_float_p, c_float_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "b2r_mlp_tc_train_bwd_film": (C.c_int, [C.c_void_p, c_float_p, c_float_p, C.c_int, C.c_int, c_ll, c_ll, c_float_p, c_float_p, C.c_void_p,
                                            C.c_void_p, C.c_size_t, c_float_p, c_float_p, c_float_p, C.c_void_p]),
    "b2r_mc_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "b2r_mc_count": (C.c_int, [c_float_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2r_mc_emit": (C.c_int, [c_float_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                              C.c_void_p, c_float_p, C.c_void_p, C.c_void_p]),
    "b2r_mc_normals": (C.c_int, [c_float_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, c_float_p, C.c_void_p]),
    "b2r_band_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "b2r_band_select": (C.c_int, [c_float_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p]),
    "b2r_lattice_rows": (C.c_int, [C.POINTER(MlpInput), C.c_void_p, c_ll, c_float_p, C.c_void_p]),
    "b2r_mc_count_band": (C.c_int, [c_float_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p]),
    "b2r_mesh_cc_scratch_bytes": (C.c_size_t, [c_ll, c_ll]),
    "b2r_mesh_cc_label": (C.c_int, [C.c_void_p, c_ll, c_ll, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2r_mesh_cc_select": (C.c_int, [C.c_void_p, c_ll, c_ll, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2r_mesh_cc_compact": (C.c_int, [c_float_p, c_float_p, C.c_void_p, c_ll, c_ll, C.c_void_p, c_float_p, c_float_p, C.c_void_p,
                                      C.c_void_p]),
    "b2r_mesh_adj_scratch_bytes": (C.c_size_t, [c_ll, c_ll]),
    "b2r_mesh_adjacency": (C.c_int, [C.c_void_p, c_ll, c_ll, C.c_void_p, C.c_void_p]),
    "b2r_mesh_smooth": (C.c_int, [c_float_p, c_ll, c_ll, C.c_int, C.c_void_p, c_float_p, C.c_void_p]),
    "b2r_mesh_normals": (C.c_int, [c_float_p, c_ll, c_ll, C.c_void_p, c_float_p, C.c_void_p]),
    "b2r_mesh_decimate_scratch_bytes": (C.c_size_t, [c_ll, c_ll]),
    "b2r_mesh_quadrics": (C.c_int, [c_float_p, c_ll, c_ll, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2r_mesh_decimate_round": (C.c_int, [c_float_p, C.c_void_p, c_ll, c_ll, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p]),
    "b2r_mesh_decimate_compact": (C.c_int, [c_float_p, C.c_void_p, C.c_void_p, c_ll, c_ll, C.c_void_p, C.c_void_p, C.c_void_p,
                                            c_float_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2r_mesh_atlas_uvs": (C.c_int, [c_ll, C.c_int, c_float_p, C.c_void_p]),
    "b2r_mesh_atlas_rows": (C.c_int, [c_float_p, c_float_p, C.c_void_p, c_ll, C.c_int, c_ll, c_ll, c_float_p, C.c_void_p]),
    "b2r_mesh_atlas_texture": (C.c_int, [c_float_p, c_ll, C.c_int, c_ll, c_ll, C.c_void_p, C.c_void_p]),
}

_lock = threading.Lock()
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: the CUDA library is the product and there is no fallback. "
                        "Build it with `make -C msra_practice_project_b200/csrc` (or __graft_entry__.build()).")
                handle = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(handle, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().b2r_last_error()
        raise RuntimeError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None passes NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr(device=None) -> int:
    import torch
    return torch.cuda.current_stream(device).cuda_stream
