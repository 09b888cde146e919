"""ctypes binding of libsqmc_b200.so (the C ABI in include/sqmc_b200.h).

There is no fallback: if the shared library is missing or no sm_100 GPU is
usable, every call raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libsqmc_b200.so")
_lib = None

# every symbol include/sqmc_b200.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "sqmc_b200_get_unique_id", "sqmc_b200_init", "sqmc_b200_finalize", "sqmc_b200_last_error",
    "sqmc_b200_system_chem", "sqmc_b200_system_heg", "sqmc_b200_system_hubbardk", "sqmc_b200_free",
    "sqmc_b200_build_h", "sqmc_b200_export_upper", "sqmc_b200_import_upper", "sqmc_b200_nnz",
    "sqmc_b200_local_rows", "sqmc_b200_diagonal", "sqmc_b200_matvec", "sqmc_b200_projector",
    "sqmc_b200_scale_values", "sqmc_b200_set_row_bundle", "sqmc_b200_lanczos", "sqmc_b200_davidson_single", "sqmc_b200_pt2", "sqmc_b200_pt2_sample", "sqmc_b200_pt2_alias", "sqmc_b200_davidson", "sqmc_b200_matvec_dev", "sqmc_b200_device_malloc",
    "sqmc_b200_device_free", "sqmc_b200_memcpy_h2d", "sqmc_b200_memcpy_d2h", "sqmc_b200_device_sync",
    "sqmc_b200_get_perm", "sqmc_b200_build_times", "sqmc_b200_launch_count", "sqmc_b200_partition_rows", "sqmc_b200_get_row", "sqmc_b200_system_orbital_symmetries", "sqmc_b200_hci_select",
    "sqmc_b200_hci_new_dets", "sqmc_b200_set_hf_to_psit",
    "sqmc_b200_set_ownership", "sqmc_b200_matvec_local", "sqmc_b200_projector_local", "sqmc_b200_davidson_local",
    "sqmc_b200_last_build_incremental", "sqmc_b200_alloc_stall_ms", "sqmc_b200_register_host", "sqmc_b200_unregister_host", "sqmc_b200_exchange_mode",
    "sqmc_b200_one_rdm", "sqmc_b200_two_rdm", "sqmc_b200_orbital_derivatives", "sqmc_b200_sigma",
    "sqmc_b200_orbital_gradient_response", "sqmc_b200_ladder", "sqmc_b200_ladder_result", "sqmc_b200_lanczos_tridiagonal",
    "sqmc_b200_transition_one_rdm", "sqmc_b200_transition_two_rdm",
]


class SqmcError(RuntimeError):
    pass


def so_path():
    return _SO


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise SqmcError("libsqmc_b200.so not built (run `python -m sqmc_b200.build`); there is no CPU fallback")
    L = C.CDLL(_SO, mode=C.RTLD_GLOBAL)
    vp, i32, i64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double
    L.sqmc_b200_last_error.restype = C.c_char_p
    L.sqmc_b200_launch_count.restype = i64
    L.sqmc_b200_alloc_stall_ms.restype = dbl
    L.sqmc_b200_alloc_stall_ms.argtypes = [i32]
    L.sqmc_b200_get_unique_id.argtypes = [vp]
    L.sqmc_b200_init.argtypes = [i32, i32, i32, vp]
    L.sqmc_b200_system_chem.argtypes = [vp, i32, i32, i32, vp, i64, vp, i32, i32]
    L.sqmc_b200_system_heg.argtypes = [vp, i32, i32, vp, dbl, i32, i32]
    L.sqmc_b200_system_hubbardk.argtypes = [vp, i32, i32, vp, vp, dbl, i32, i32]
    L.sqmc_b200_free.argtypes = [vp]
    L.sqmc_b200_build_h.argtypes = [vp, i64, vp, vp, i64, vp]
    L.sqmc_b200_export_upper.argtypes = [vp, vp, vp, vp]
    L.sqmc_b200_import_upper.argtypes = [vp, i64, vp, vp, vp]
    L.sqmc_b200_nnz.argtypes = [vp, vp, vp, vp]
    L.sqmc_b200_local_rows.argtypes = [vp, vp, vp]
    L.sqmc_b200_diagonal.argtypes = [vp, i64, vp, vp, vp]
    L.sqmc_b200_matvec.argtypes = [vp, vp, vp, i32, i64]
    L.sqmc_b200_projector.argtypes = [vp, dbl, dbl, vp, vp]
    L.sqmc_b200_scale_values.argtypes = [vp, dbl]
    L.sqmc_b200_set_row_bundle.argtypes = [vp, i32]
    L.sqmc_b200_one_rdm.argtypes = [vp, i64, vp, vp, i32, vp, i64, vp]
    L.sqmc_b200_two_rdm.argtypes = [vp, i64, vp, vp, i32, vp, i64, vp]
    L.sqmc_b200_transition_one_rdm.argtypes = [vp, i64, vp, vp, i32, vp, vp, i64, vp]
    L.sqmc_b200_transition_two_rdm.argtypes = [vp, i64, vp, vp, i32, vp, vp, i64, vp]
    L.sqmc_b200_orbital_derivatives.argtypes = [vp, i64, vp, vp, i32, vp, i64, vp, vp, vp, vp]
    L.sqmc_b200_sigma.argtypes = [vp, i64, vp, vp, i32, vp, i64, vp, vp]
    L.sqmc_b200_orbital_gradient_response.argtypes = [vp, i64, vp, vp, i32, vp, vp, i64, vp, vp]
    L.sqmc_b200_ladder.argtypes = [vp, i64, vp, vp, i32, vp, i64, i32, i32, i32, i32, vp, vp]
    L.sqmc_b200_ladder_result.argtypes = [vp, vp, vp, vp, i64]
    L.sqmc_b200_lanczos_tridiagonal.argtypes = [vp, i32, vp, i64, i32, dbl, vp, vp, vp, vp]
    L.sqmc_b200_pt2.argtypes = [vp, i64, vp, vp, vp, dbl, dbl, vp, vp]
    L.sqmc_b200_pt2_sample.argtypes = [vp, i64, vp, vp, i64, vp, vp, vp, vp, i32, dbl, dbl, dbl, vp, vp]
    L.sqmc_b200_pt2_alias.argtypes = [vp, i64, vp, vp, vp, dbl, dbl, dbl, i32, dbl, vp, i32, vp, vp, vp, vp, vp]
    L.sqmc_b200_davidson_single.argtypes = [vp, vp, vp, vp, dbl, i32, vp, vp, i32, vp]
    L.sqmc_b200_lanczos.argtypes = [vp, vp, vp, vp, dbl, i32, vp, vp, i32, vp]
    L.sqmc_b200_davidson.argtypes = [vp, i32, vp, vp, vp, dbl, i32, vp, vp, i32, vp]
    L.sqmc_b200_matvec_dev.argtypes = [vp, vp, vp, vp]
    L.sqmc_b200_device_malloc.argtypes = [vp, i64]
    L.sqmc_b200_device_free.argtypes = [vp]
    L.sqmc_b200_memcpy_h2d.argtypes = [vp, vp, i64]
    L.sqmc_b200_memcpy_d2h.argtypes = [vp, vp, i64]
    L.sqmc_b200_get_perm.argtypes = [vp, vp]
    L.sqmc_b200_build_times.argtypes = [vp, vp]
    L.sqmc_b200_partition_rows.argtypes = [vp, i64, i32, vp]
    L.sqmc_b200_get_row.argtypes = [vp, i64, i64, vp, vp, vp]
    L.sqmc_b200_system_orbital_symmetries.argtypes = [vp, vp]
    L.sqmc_b200_hci_select.argtypes = [vp, i64, vp, vp, vp, vp, dbl, vp]
    L.sqmc_b200_hci_new_dets.argtypes = [vp, vp, vp]
    L.sqmc_b200_set_hf_to_psit.argtypes = [vp, i32]
    L.sqmc_b200_set_ownership.argtypes = [vp, vp, vp]
    L.sqmc_b200_matvec_local.argtypes = [vp, vp, vp, i32, i64]
    L.sqmc_b200_projector_local.argtypes = [vp, dbl, dbl, vp, vp]
    L.sqmc_b200_davidson_local.argtypes = [vp, i32, vp, vp, vp, dbl, i32, vp, vp, i32, vp]
    L.sqmc_b200_register_host.argtypes = [vp, i64]
    L.sqmc_b200_unregister_host.argtypes = [vp]
    L.sqmc_b200_exchange_mode.argtypes = [vp]
    L.sqmc_b200_last_build_incremental.argtypes = [vp]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise SqmcError("libsqmc_b200: " + load().sqmc_b200_last_error().decode(errors="replace"))


_inited = False


def init(device=0, rank=0, nranks=1, unique_id=None):
    """sqmc_b200_init once per process."""
    global _inited
    if _inited:
        return
    L = load()
    buf = None
    if nranks > 1:
        if unique_id is None or len(unique_id) != 128:
            raise SqmcError("init: nranks>1 needs the 128-byte ncclUniqueId from get_unique_id() on rank 0")
        buf = C.create_string_buffer(bytes(unique_id), 128)
    check(L.sqmc_b200_init(device, rank, nranks, buf))
    _inited = True


def get_unique_id():
    buf = C.create_string_buffer(128)
    check(load().sqmc_b200_get_unique_id(buf))
    return buf.raw


def finalize():
    global _inited
    if _inited:
        load().sqmc_b200_finalize()
        _inited = False
