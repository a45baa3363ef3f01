"""ctypes binding of the C ABI declared in include/joltqc_b200.h (libjoltqc_b200.so, in-tree).

The library is the product: if it is missing this module raises — there is no fallback.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# JQC_LIB_PATH selects another build of the same library (A/B experiments with tools/tune_*.py)
LIB_PATH = os.environ.get("JQC_LIB_PATH") or os.path.join(os.path.dirname(_HERE), "libjoltqc_b200.so")

EXPORTS = [
    "jqc_engine_create", "jqc_engine_destroy", "jqc_last_error", "jqc_engine_set_shard", "jqc_q_matrix",
    "jqc_dm_from_mol", "jqc_dm_to_mol", "jqc_get_jk", "jqc_get_jk_host", "jqc_build_partial", "jqc_finalize",
    "jqc_last_stats", "jqc_set_profiling", "jqc_last_class_ms", "jqc_engine_nao", "jqc_engine_mol_nao",
    "jqc_fp64_peak_probe", "jqc_last_band_stats", "jqc_jk_energy_grad", "jqc_jk_energy_grad_uhf",
]


class BasisDesc(ctypes.Structure):
    _fields_ = [
        ("nbas", ctypes.c_int),
        ("records", ctypes.POINTER(ctypes.c_double)),
        ("angs", ctypes.POINTER(ctypes.c_int)),
        ("nprims", ctypes.POINTER(ctypes.c_int)),
        ("ao_loc", ctypes.POINTER(ctypes.c_int)),
        ("pad", ctypes.POINTER(ctypes.c_uint8)),
        ("ngroups", ctypes.c_int),
        ("group_offset", ctypes.POINTER(ctypes.c_int)),
        ("mol_ao_offset", ctypes.POINTER(ctypes.c_int)),
        ("mol_nao", ctypes.c_int),
        ("mol_cart", ctypes.c_int),
        ("c2s", ctypes.POINTER(ctypes.c_double)),
    ]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m joltqc_b200.build` "
            "(joltqc_b200 has no CPU or PyTorch fallback for the J/K path)")
    L = ctypes.CDLL(LIB_PATH)
    vp, dp, ci, cd = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    L.jqc_last_error.restype = ctypes.c_char_p
    L.jqc_engine_create.argtypes = [ctypes.POINTER(BasisDesc), ci, ctypes.POINTER(vp)]
    L.jqc_engine_destroy.argtypes = [vp]
    L.jqc_engine_destroy.restype = None
    L.jqc_engine_set_shard.argtypes = [vp, ci, ci]
    L.jqc_q_matrix.argtypes = [vp, cd, ctypes.POINTER(vp)]
    L.jqc_dm_from_mol.argtypes = [vp, dp, ci, dp, vp]
    L.jqc_dm_to_mol.argtypes = [vp, dp, ci, dp, vp]
    L.jqc_get_jk.argtypes = [vp, dp, ci, ci, ci, ci, cd, cd, cd, dp, dp, vp]
    L.jqc_get_jk_host.argtypes = [vp, dp, ci, ci, ci, ci, cd, cd, cd, dp, dp]
    L.jqc_build_partial.argtypes = [vp, dp, ci, ci, ci, ci, cd, cd, cd, ctypes.POINTER(vp),
                                    ctypes.POINTER(ctypes.c_size_t), vp]
    L.jqc_finalize.argtypes = [vp, dp, dp, vp]
    L.jqc_jk_energy_grad.argtypes = [vp, dp, cd, cd, cd, cd, ctypes.POINTER(ci), ci, dp,
                                     ctypes.POINTER(ctypes.c_longlong), vp]
    L.jqc_jk_energy_grad_uhf.argtypes = [vp, dp, cd, cd, cd, cd, ctypes.POINTER(ci), ci, dp,
                                         ctypes.POINTER(ctypes.c_longlong), vp]
    L.jqc_last_stats.argtypes = [vp, ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_longlong),
                                 ctypes.POINTER(ci)]
    L.jqc_last_band_stats.argtypes = [vp, ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_float)]
    L.jqc_set_profiling.argtypes = [vp, ci]
    L.jqc_last_class_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_float)]
    L.jqc_engine_nao.argtypes = [vp]
    L.jqc_engine_mol_nao.argtypes = [vp]
    L.jqc_fp64_peak_probe.argtypes = [ci, ctypes.POINTER(cd), ctypes.POINTER(cd)]
    _lib = L
    return L


class JQCError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        msg = load().jqc_last_error()
        raise JQCError(f"joltqc_b200 error {rc}: {msg.decode() if msg else ''}")
