"""Python face of the CPU oracle of the J/K energy gradient (tests/grad_oracle.c).

The library is compiled on first use with the flags of oracle/Makefile into a per-user cache directory
outside the tree (keyed by the hash of the sources), so that the pinned oracle/ stays untouched.
"""
import ctypes
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SRC = os.path.join(_HERE, "grad_oracle.c")
CFLAGS = ["-O2", "-fopenmp", "-fPIC", "-std=gnu11", "-Wall", "-Wno-unused-variable", "-Wno-unused-function",
          "-ffp-contract=off"]
_LIB = None


def build():
    h = hashlib.sha256()
    for f in (_SRC, os.path.join(_ORACLE, "jk_oracle.c"), os.path.join(_ORACLE, "rys_tables.h")):
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(CFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), f"joltqc_grad_oracle_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"libgradoracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = so + f".{os.getpid()}.tmp"
        subprocess.run(["gcc"] + CFLAGS + ["-I", _ORACLE, "-shared", "-o", tmp, _SRC, "-lm"], check=True)
        os.replace(tmp, so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        dp, ip, fp = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_float)
        L.grad_oracle_eri_block.argtypes = [dp, ip, ip] + [ctypes.c_int] * 4 + [ctypes.c_double, dp]
        L.oracle_jk_grad.restype = ctypes.c_long
        L.oracle_jk_grad.argtypes = [ctypes.c_int, dp, ip, ip, ip, fp, fp, ctypes.c_float, dp, ctypes.c_double,
                                     ctypes.c_double, ctypes.c_double, ctypes.c_float, dp]
        _LIB = L
    return _LIB


def _p(a, t):
    return a.ctypes.data_as(ctypes.POINTER(t))


def eri_block(orc, i, j, k, l, omega=0.0):
    """(ij|kl) of the l <= 5 twin of the pinned eri_block, on the shell table of an oracle.OracleJK."""
    n = [(int(orc.angs[s]) + 1) * (int(orc.angs[s]) + 2) // 2 for s in (i, j, k, l)]
    out = np.zeros(n)
    lib().grad_oracle_eri_block(_p(orc.rec, ctypes.c_double), _p(orc.angs, ctypes.c_int), _p(orc.nprims, ctypes.c_int),
                                i, j, k, l, float(omega or 0.0), _p(out, ctypes.c_double))
    return out


def jk_energy_grad(orc, dm, j_factor=1.0, k_factor=1.0, omega=None, cutoff=1e-13):
    """Nuclear gradient of E_jk = (j_factor/2) tr(D J[D]) - (k_factor/4) tr(D K[D]) for one symmetric density
    in the molecule's AO basis (J, K of get_jk(dm, hermi=1, omega=omega)), with the AO transform, density
    pooling and Schwarz matrix of the pinned oracle ``orc`` (oracle.OracleJK).  Returns the (natm, 3)
    gradient and the number of quartets evaluated."""
    dm = np.asarray(dm, dtype=np.float64)
    T = orc.transform()
    d = np.ascontiguousarray(T @ dm @ T.T)
    log_dm, log_max = orc.dm_cond(d[None], 1)
    q = orc.q_matrix(omega)
    gsh = np.zeros((orc.nbas, 3))
    nq = lib().oracle_jk_grad(orc.nbas, _p(orc.rec, ctypes.c_double), _p(orc.angs, ctypes.c_int),
                              _p(orc.nprims, ctypes.c_int), _p(orc.ao_loc, ctypes.c_int), _p(q, ctypes.c_float),
                              _p(log_dm, ctypes.c_float), ctypes.c_float(log_max), _p(d, ctypes.c_double),
                              float(j_factor), float(k_factor), float(omega or 0.0),
                              ctypes.c_float(np.float32(math.log(cutoff))), _p(gsh, ctypes.c_double))
    atom = np.asarray(orc.layout.shell_atom)
    g = np.zeros((orc.layout._mol.natm, 3))
    np.add.at(g, atom[atom >= 0], gsh[atom >= 0])
    return g, int(nq)
