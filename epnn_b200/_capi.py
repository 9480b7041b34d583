"""ctypes binding of libepnn_b200.so (include/epnn_b200.h).  No torch types cross this boundary.

The library is built in-tree by ``__graft_entry__.build()``.  There is no CPU fallback: if the shared
object is missing, ``load()`` raises; if no CUDA device is usable, ``epnn_create`` fails."""
from __future__ import annotations

import ctypes as C
import os

_LIB = None
# EPNN_B200_LIB: development override (A/B of kernel variants built by tools/build_variant.sh); the product is the in-tree library
LIB_PATH = os.environ.get("EPNN_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libepnn_b200.so")

EPNN_OK = 0
ERRORS = {-1: "EPNN_E_INVALID", -2: "EPNN_E_CUDA", -3: "EPNN_E_NOMEM", -4: "EPNN_E_CAPACITY", -5: "EPNN_E_UNSUPPORTED"}


class EpnnError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"{ERRORS.get(code, code)}: {msg}")
        self.code = code


class Stats(C.Structure):
    _fields_ = [("n_systems", C.c_int64), ("n_atoms", C.c_int64), ("n_pairs_e", C.c_int64), ("n_pairs_near", C.c_int64),
                ("n_row_groups", C.c_int64), ("n_chunks", C.c_int64), ("n_launches", C.c_int64),
                ("ms_total", C.c_float), ("ms_h2d", C.c_float), ("ms_neighbor", C.c_float), ("ms_gnn_pair", C.c_float),
                ("ms_gnn_atom", C.c_float), ("ms_epn_pair", C.c_float), ("ms_epn_atom", C.c_float), ("ms_d2h", C.c_float),
                ("n_far_dedup_rows", C.c_int64), ("n_gnn_near_slots", C.c_int64), ("n_gnn_far_slots", C.c_int64),
                ("precision_used", C.c_int32), ("probe_err32", C.c_float), ("probe_err48", C.c_float),
                ("atom_tensor_used", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}



# name -> (restype, argtypes); mirrors include/epnn_b200.h one to one
SIGNATURES = {
    "epnn_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "epnn_destroy": (None, [C.c_void_p]),
    "epnn_last_error": (C.c_char_p, [C.c_void_p]),
    "epnn_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_double]),
    "epnn_infer_batch": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "epnn_infer_batch_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "epnn_electrostatics": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "epnn_electrostatics_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "epnn_potential_points": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]),
    "epnn_potential_points_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]),
    "epnn_neighbors": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_int64, C.POINTER(C.c_int64)]),
    "epnn_init_edges": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "epnn_infer_dense": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p]),
    "epnn_get_hidden": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "epnn_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "epnn_host_free": (C.c_int, [C.c_void_p]),
    "epnn_shard_unique_id": (C.c_int, [C.c_void_p]),
    "epnn_shard_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "epnn_shard_slice": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "epnn_shard_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "epnn_get_stream": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "epnn_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "epnn_measure_fp32_peak": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double)]),
    "epnn_xyz_load": (C.c_int, [C.POINTER(C.c_char_p), C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "epnn_xyz_parse_text": (C.c_int, [C.c_char_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "epnn_xyz_n_systems": (C.c_int64, [C.c_void_p]),
    "epnn_xyz_n_atoms": (C.c_int64, [C.c_void_p]),
    "epnn_xyz_offsets": (C.c_void_p, [C.c_void_p]),
    "epnn_xyz_coords": (C.c_void_p, [C.c_void_p]),
    "epnn_xyz_species": (C.c_void_p, [C.c_void_p]),
    "epnn_xyz_charges": (C.c_void_p, [C.c_void_p]),
    "epnn_xyz_error": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "epnn_xyz_error_message": (C.c_char_p, [C.c_void_p]),
    "epnn_xyz_free": (None, [C.c_void_p]),
    "epnn_rbf_centers": (C.c_int, [C.c_void_p]),
    "epnn_rbf_basis": (C.c_int, [C.c_void_p]),
    "epnn_version": (C.c_char_p, []),
}


def load():
    """dlopen the in-tree library and declare every prototype.  Raises if the library is missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = os.environ.get("EPNN_B200_LIB", LIB_PATH)      # development hook: try an alternative build of the same ABI
    if not os.path.exists(path):
        raise ImportError(f"{path} not found: run `python __graft_entry__.py` (nvcc, sm_100a) first. "
                          "epnn_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib
