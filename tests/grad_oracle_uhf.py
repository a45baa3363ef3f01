"""Python face of the CPU oracle of the spin-unrestricted J/K energy gradient (tests/grad_oracle_uhf.c).

The library is compiled on first use with the flags of tests/grad_oracle.py into the same per-user cache
directory outside the tree (keyed by the hash of the sources), so that the pinned oracle/ stays untouched.
"""
import ctypes
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

from tests.grad_oracle import CFLAGS

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SRC = os.path.join(_HERE, "grad_oracle_uhf.c")
_LIB = None


def build():
    h = hashlib.sha256()
    for f in (_SRC, os.path.join(_HERE, "grad_oracle.c"), os.path.join(_ORACLE, "jk_oracle.c"),
              os.path.join(_ORACLE, "rys_tables.h")):
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(CFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), f"joltqc_grad_oracle_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"libgradoracle_uhf_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = so + f".{os.getpid()}.tmp"
        subprocess.run(["gcc"] + CFLAGS + ["-I", _HERE, "-I", _ORACLE, "-shared", "-o", tmp, _SRC, "-lm"], check=True)
        os.replace(tmp, so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        dp, ip, fp = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_float)
        L.oracle_jk_grad_uhf.restype = ctypes.c_long
        L.oracle_jk_grad_uhf.argtypes = [ctypes.c_int, dp, ip, ip, ip, fp, fp, fp, ctypes.c_float, dp, dp,
                                         ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_float, dp]
        _LIB = L
    return _LIB


def _p(a, t):
    return a.ctypes.data_as(ctypes.POINTER(t))


def jk_energy_grad_uhf(orc, dm, j_factor=1.0, k_factor=1.0, omega=None, cutoff=1e-13):
    """Nuclear gradient of E_U = (j_factor/2) tr(Dt J[Dt]) - (k_factor/2) [tr(Da K[Da]) + tr(Db K[Db])] for the
    symmetric spin densities ``dm = [Da, Db]`` (2, nao, nao) in the molecule's AO basis and Dt = Da + Db
    (J, K of get_jk([Da, Db], hermi=1, omega=omega)), with the AO transform, density pooling and Schwarz matrix
    of the pinned oracle ``orc`` (oracle.OracleJK).  The J term is screened on the pooled Dt (dJ), the K terms
    on max_s |Ds| (dS), the tile lists on twice the larger of the two maxima.  Returns the (natm, 3) gradient
    and the number of quartets evaluated."""
    dm = np.asarray(dm, dtype=np.float64)
    assert dm.ndim == 3 and dm.shape[0] == 2
    T = orc.transform()
    d = np.ascontiguousarray(np.stack([T @ dm[0] @ T.T, T @ dm[1] @ T.T]))
    dt = np.ascontiguousarray(d[0] + d[1])
    log_ds, max_s = orc.dm_cond(d, 1)
    log_dj, max_j = orc.dm_cond(dt[None], 1)
    log_max = max(np.float32(max_s), np.float32(max_j))
    q = orc.q_matrix(omega)
    gsh = np.zeros((orc.nbas, 3))
    nq = lib().oracle_jk_grad_uhf(orc.nbas, _p(orc.rec, ctypes.c_double), _p(orc.angs, ctypes.c_int),
                                  _p(orc.nprims, ctypes.c_int), _p(orc.ao_loc, ctypes.c_int), _p(q, ctypes.c_float),
                                  _p(log_dj, ctypes.c_float), _p(log_ds, ctypes.c_float), ctypes.c_float(log_max),
                                  _p(d, ctypes.c_double), _p(dt, ctypes.c_double), float(j_factor), float(k_factor),
                                  float(omega or 0.0), ctypes.c_float(np.float32(math.log(cutoff))),
                                  _p(gsh, ctypes.c_double))
    atom = np.asarray(orc.layout.shell_atom)
    g = np.zeros((orc.layout._mol.natm, 3))
    np.add.at(g, atom[atom >= 0], gsh[atom >= 0])
    return g, int(nq)
