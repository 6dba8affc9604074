"""ctypes binding of ``libpdbeda_b200.so`` (the C ABI declared in ``include/pdbeda_b200.h``).

There is deliberately no fallback: if the shared library is missing or a call fails, an exception is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libpdbeda_b200.so")

PE_SPHERE_NOUT = 8


class PeGeom(ctypes.Structure):
    """Mirror of ``struct pe_geom`` (include/pdbeda_b200.h)."""
    _fields_ = [
        ("ncrs", ctypes.c_int32 * 3),
        ("crs_start", ctypes.c_int32 * 3),
        ("xyz_interval", ctypes.c_int32 * 3),
        ("crs_interval", ctypes.c_int32 * 3),
        ("unique_ncrs", ctypes.c_int32 * 3),
        ("map2xyz", ctypes.c_int32 * 3),
        ("map2crs", ctypes.c_int32 * 3),
        ("orthogonal", ctypes.c_int32),
        ("mv_perm", ctypes.c_int32 * 3),
        ("mv_fma", ctypes.c_int32),
        ("grid_length", ctypes.c_double * 3),
        ("origin", ctypes.c_double * 3),
        ("ortho", ctypes.c_double * 9),
        ("deortho", ctypes.c_double * 9),
    ]


class PdbEdaLibError(RuntimeError):
    pass


_P = ctypes.c_void_p
_I32 = ctypes.c_int32
_I64 = ctypes.c_int64
_F32 = ctypes.c_float
_GEOM = ctypes.POINTER(PeGeom)

# name -> (restype, argtypes); every symbol include/pdbeda_b200.h declares
SIGNATURES = {
    "pe_abi_version": (ctypes.c_int, []),
    "pe_last_error": (ctypes.c_char_p, []),
    "pe_device_info": (ctypes.c_int, [ctypes.POINTER(_I32)] * 3),
    "pe_launch_count": (ctypes.c_longlong, []),
    "pe_profile_enable": (None, [ctypes.c_int]),
    "pe_profile_reset": (None, []),
    "pe_profile_entries": (ctypes.c_int, []),
    "pe_profile_get": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_longlong),
                                      ctypes.POINTER(ctypes.c_double)]),
    "pe_stats_workspace_bytes": (_I64, []),
    "pe_map_mean_std": (ctypes.c_int, [_P, _I64, _P, _P, _P]),
    "pe_map_sum_abs": (ctypes.c_int, [_P, _I64, _F32, _P, _P, _P]),
    "pe_sum_abs_f64": (ctypes.c_int, [_P, _I64, _F32, _P, _P, _P]),
    "pe_point_density": (ctypes.c_int, [_GEOM, _P, _I64, _P, _P, _P, _P]),
    "pe_xyz2crs": (ctypes.c_int, [_GEOM, _I64, _P, _P, _P]),
    "pe_crs2xyz": (ctypes.c_int, [_GEOM, _I64, _P, _P, _P]),
    "pe_sphere_workspace_bytes": (_I64, [_I64]),
    "pe_sphere_union_warp_cycles": (ctypes.c_int, [ctypes.POINTER(ctypes.c_ulonglong)]),
    "pe_sphere_sums": (ctypes.c_int, [_GEOM, _P, _I32, _P, _P, _I32, _P, _F32, _F32, _P, _P, _P]),
    "pe_sphere_sums_atoms_and_groups": (ctypes.c_int, [_GEOM, _P, _I32, _P, _P, _F32, _P, _I32, _P, _F32, _F32, _P, _P, _P, _P]),
    "pe_sphere_count": (ctypes.c_int, [_GEOM, _P, _I32, _P, _P, _F32, _P, _P, _P]),
    "pe_sphere_fill": (ctypes.c_int, [_GEOM, _P, _I32, _P, _P, _F32, _P, _I32, _P, _P, _P, _P]),
    "pe_blob_workspace_bytes": (_I64, [_GEOM, _I64]),
    "pe_blob_stage_times": (ctypes.c_int, [ctypes.POINTER(ctypes.c_ulonglong)]),
    "pe_blob_label": (ctypes.c_int, [_GEOM, _P, _F32, _F32, _I64, _I64, _P, _P, _P, _P, _P, _P, _P]),
    "pe_cluster_workspace_bytes": (_I64, [_I64]),
    "pe_cluster_crs": (ctypes.c_int, [_I64, _P, _P, _P, _P, _P]),
    "pe_cluster_crs_grouped": (ctypes.c_int, [_I64, _P, _P, _P, _P, _P, _P, _P]),
    "pe_crs_stats": (ctypes.c_int, [_GEOM, _P, _I64, _P, _P, _P, _I64, _P, _P]),
    "pe_pair_metrics": (ctypes.c_int, [_GEOM, _P, _P, _I64, _P, _P, _P, _I64, _P, _P]),
    "pe_pair_union_workspace_bytes": (_I64, [_I32]),
    "pe_pair_union_metrics": (ctypes.c_int, [_I32, _P, _I32, _P, _P, _P, _P, _P, _P, _P]),
    "pe_overlap_workspace_bytes": (_I64, [_I64, _I64]),
    "pe_overlap_pairs": (ctypes.c_int, [_I64, _P, _P, _P, _I64, _P, _P, _P, _P]),
    "pe_symmetry_workspace_bytes": (_I64, [_I32, _I32]),
    "pe_symmetry_expand": (ctypes.c_int, [_GEOM, _I32, _P, _I32, _P, _P, ctypes.POINTER(ctypes.c_double),
                                          ctypes.POINTER(ctypes.c_double), _I64, _P, _P, _P, _P, _P, _P]),
    "pe_nearest_atom": (ctypes.c_int, [_I64, _P, _I64, _P, _P, _P, _P]),
    "pe_slab_exchange_bytes": (_I64, [_I64, _I64]),
    "pe_slab_workspace_bytes": (_I64, [_I32, _I64, _I32, _I32]),
    "pe_slab_boundary": (ctypes.c_int, [_GEOM, _I32, _I32, _I32, _P, _I64, _P, _P, _I64, _I64, _P, _P, _P]),
    "pe_slab_merge": (ctypes.c_int, [_I32, _I32, _P, _I64, _I64, _I32, _I32, _P, _P, _P, _P]),
    "pe_slab_relabel": (ctypes.c_int, [_GEOM, _I32, _I32, _P, _I64, _P, _P, _P, _I64, _P, _P, _I64, _P, _P, _P]),
    "pe_slab_status": (ctypes.c_int, [_P, _P, ctypes.POINTER(_I32)]),
    "pe_cloud_workspace_bytes": (_I64, [_I64, _I64, _I64, _I64]),
    "pe_cloud_count": (ctypes.c_int, [_I32, _P, _I32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pe_cloud_aggregate": (ctypes.c_int, [_I32, _P, _I32, _P, _P, _P, _P, _P, _P, _P, _I32, _P, _I64, _I32, ctypes.c_double, _P, _P, _P,
                                          _P, _P]),
    "pe_cloud_status": (ctypes.c_int, [_P, _P, ctypes.POINTER(_I32)]),
    "pe_cloud_statistics": (ctypes.c_int, [_I32, _P, _I32, _P, _P, _P, _P, _I32, _P, _P, _P, _P, _I32, _P, _P, ctypes.c_double, _P, _P,
                                           _P, _P]),
}

_lib = None


def load():
    """Loads the shared library (once) and declares every prototype.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise PdbEdaLibError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
            "`make -C pdb_eda_b200/csrc` (there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.pe_abi_version() != 1:
        raise PdbEdaLibError("libpdbeda_b200.so ABI version %d, expected 1" % lib.pe_abi_version())
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().pe_last_error()
        raise PdbEdaLibError("%s failed (%d): %s" % (what, rc, msg.decode("utf-8", "replace") if msg else "?"))


def require_device():
    """Raises unless a CUDA device is usable through the library; returns (sm_count, cc_major, cc_minor)."""
    lib = load()
    sm, major, minor = _I32(0), _I32(0), _I32(0)
    check(lib.pe_device_info(ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor)), "pe_device_info")
    return sm.value, major.value, minor.value


def profile(enable=None, reset=False):
    """Kernel-level device timing of the library.  ``profile(True)`` / ``profile(False)`` switch it on and off;
    ``profile()`` returns {kernel name: (launches, total ms)} accumulated since the last reset."""
    lib = load()
    if reset:
        lib.pe_profile_reset()
    if enable is not None:
        lib.pe_profile_enable(1 if enable else 0)
        return None
    out = {}
    for i in range(lib.pe_profile_entries()):
        name, count, ms = ctypes.c_char_p(), ctypes.c_longlong(0), ctypes.c_double(0.0)
        if lib.pe_profile_get(i, ctypes.byref(name), ctypes.byref(count), ctypes.byref(ms)) == 0:
            out[name.value.decode()] = (count.value, ms.value)
    return out


def launch_count():
    return load().pe_launch_count()
