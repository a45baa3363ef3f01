"""Shell table construction for the J/K engine (host side, numpy only).

Mirrors the reference interface ``jqc/pyscf/basis.py`` for the J/K path:
``split_basis`` (:678-837), ``sort_group_basis`` (:483-675), ``BasisLayout`` (:66-480) and
``compute_q_matrix`` (:840-867) — same names, argument meaning and resulting table
semantics — but the implementation is written against plain ``_atm/_bas/_env`` arrays
(PySCF optional), is vectorised per group, and leaves every device-side job (Schwarz
matrix, AO transforms) to the CUDA engine behind the C ABI (include/joltqc_b200.h).

Table semantics kept from the reference (SURVEY appendix B):
  * generally-contracted shells are decontracted, shells with more than NPRIM_MAX
    primitives are split into chunks that alias the same molecular AOs;
  * shells are grouped by (l, nprim), groups ordered by l ascending / nprim descending,
    each group padded to a multiple of ``alignment`` with copies of its first shell;
    pads have zero AO width and Schwarz value -100;
  * packed record per shell: [x, y, z, ao_loc, c0, e0, c1, e1, c2, e2, 0, 0];
  * s and p coefficients carry sqrt((2l+1)/4pi).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from ..constants import BASIS_STRIDE, LMAX, NPRIM_MAX

# libcint _bas / _atm columns (jqc/pyscf/basis.py:519-528)
ATOM_OF, ANG_OF, NPRIM_OF, NCTR_OF, KAPPA_OF, PTR_EXP, PTR_COEFF = 0, 1, 2, 3, 4, 5, 6
PTR_COORD = 1

__all__ = ["BasisLayout", "compute_q_matrix", "sort_group_basis", "split_basis", "SplitMol"]


@dataclass
class SplitMol:
    """The decontracted + split shell list in libcint layout (what the reference keeps as an
    un-built ``pyscf.gto.Mole``, basis.py:831-837)."""
    _atm: np.ndarray
    _bas: np.ndarray
    _env: np.ndarray
    cart: bool

    @property
    def nbas(self):
        return int(self._bas.shape[0])


def split_basis(mol):
    """Decontract (nctr > 1) and split (nprim > NPRIM_MAX) every shell of ``mol``.

    Returns (SplitMol, split_to_decontracted) where the map gives, for each resulting
    shell, the index of its parent in the fully decontracted shell list (one entry per
    (shell, contraction)) — the chunks of a split shell share one parent and therefore the
    same molecular AOs (reference: basis.py:678-837)."""
    bas = np.asarray(mol._bas)
    env = list(np.asarray(mol._env, dtype=np.float64))
    rows, parent = [], []
    dec = 0
    for b in bas:
        nprim, nctr = int(b[NPRIM_OF]), int(b[NCTR_OF])
        e0, c0 = int(b[PTR_EXP]), int(b[PTR_COEFF])
        for ic in range(nctr):
            cptr = c0 + ic * nprim
            if nprim <= NPRIM_MAX:
                row = b.copy()
                row[NCTR_OF] = 1
                row[PTR_COEFF] = cptr
                rows.append(row)
                parent.append(dec)
            else:
                for p0 in range(0, nprim, NPRIM_MAX):
                    n = min(NPRIM_MAX, nprim - p0)
                    row = b.copy()
                    row[NPRIM_OF], row[NCTR_OF] = n, 1
                    row[PTR_EXP], row[PTR_COEFF] = e0 + p0, cptr + p0
                    rows.append(row)
                    parent.append(dec)
            dec += 1
    sm = SplitMol(np.asarray(mol._atm).copy(), np.asarray(rows, dtype=np.int32).reshape(-1, bas.shape[1]),
                  np.asarray(env), bool(mol.cart))
    return sm, np.asarray(parent, dtype=np.int32)


def sort_group_basis(mol, alignment=4, dtype=np.float64):
    """Group the (already decontracted) shells of ``mol`` by (l, nprim) and pad.

    Returns ((ce, coords, angs, nprims), to_split_map, pad_id, (group_key, group_offset))
    with the reference's meaning (basis.py:483-675).  ``ce`` is (n, BASIS_STRIDE-4) with
    interleaved (coefficient, exponent) pairs, unused slots zero."""
    bas, env, atm = np.asarray(mol._bas), np.asarray(mol._env), np.asarray(mol._atm)
    if np.any(bas[:, NCTR_OF] != 1):
        raise AssertionError("sort_group_basis expects a decontracted shell list (nctr == 1)")
    keys = sorted({(int(b[ANG_OF]), int(b[NPRIM_OF])) for b in bas}, key=lambda k: (k[0], -k[1]))
    ce_l, xyz_l, map_l, pad_l, ang_l, np_l, offs = [], [], [], [], [], [], [0]
    for l, nprim in keys:
        idx = np.nonzero((bas[:, ANG_OF] == l) & (bas[:, NPRIM_OF] == nprim))[0]
        npad = (-len(idx)) % alignment
        sel = np.concatenate([idx, np.full(npad, idx[0], dtype=idx.dtype)])
        fac = math.sqrt((2 * l + 1) / (4.0 * math.pi)) if l < 2 else 1.0
        ce = np.zeros((len(sel), BASIS_STRIDE - 4), dtype=dtype)
        for p in range(nprim):
            ce[:, 2 * p] = env[bas[sel, PTR_COEFF] + p] * fac
            ce[:, 2 * p + 1] = env[bas[sel, PTR_EXP] + p]
        xyz = np.zeros((len(sel), 4), dtype=np.float64)
        cptr = atm[bas[sel, ATOM_OF], PTR_COORD]
        for d in range(3):
            xyz[:, d] = env[cptr + d]
        ce_l.append(ce)
        xyz_l.append(xyz)
        map_l.append(sel.astype(np.int32))
        pad_l.append(np.arange(len(sel)) >= len(idx))
        ang_l.append(np.full(len(sel), l, dtype=np.int32))
        np_l.append(np.full(len(sel), nprim, dtype=np.int32))
        offs.append(offs[-1] + len(sel))
    bas_info = (np.concatenate(ce_l), np.concatenate(xyz_l).astype(dtype), np.concatenate(ang_l), np.concatenate(np_l))
    return bas_info, np.concatenate(map_l), np.concatenate(pad_l), (np.asarray(keys, dtype=np.int32), np.asarray(offs))


@dataclass
class BasisLayout:
    ce: np.ndarray          # (nbasis, BASIS_STRIDE-4)
    coords: np.ndarray      # (nbasis, 4)
    angs: np.ndarray        # (nbasis,) int32
    nprims: np.ndarray      # (nbasis,) int32
    to_split_map: np.ndarray
    pad_id: np.ndarray
    group_key: np.ndarray   # (ngroups, 2) [l, nprim]
    group_offset: np.ndarray
    dtype: np.dtype
    alignment: int = 4
    _mol: Optional[object] = None
    _splitted_mol: Optional[SplitMol] = None
    _split_to_decontracted: Optional[np.ndarray] = None
    _cache: dict = field(default_factory=dict, repr=False)

    # ------------------------------------------------------------------ construction
    @classmethod
    def from_mol(cls, mol, alignment: int = 4, dtype=np.float64) -> "BasisLayout":
        sm, parent = split_basis(mol)
        (ce, coords, angs, nprims), to_split, pad, (gkey, goff) = sort_group_basis(sm, alignment, dtype)
        if angs[~pad].size and int(angs[~pad].max()) > LMAX:
            raise AssertionError(f"Angular momentum {int(angs[~pad].max())} exceeds maximum supported value of {LMAX}")
        return cls(ce=ce, coords=coords, angs=angs, nprims=nprims, to_split_map=to_split, pad_id=pad,
                   group_key=gkey, group_offset=goff, dtype=np.dtype(dtype), alignment=alignment,
                   _mol=mol, _splitted_mol=sm, _split_to_decontracted=parent)

    # ------------------------------------------------------------------ accessors
    @property
    def bas_info(self):
        return (self.ce, self.coords, self.angs, self.nprims)

    @property
    def group_info(self):
        return (self.group_key, self.group_offset)

    @property
    def nbasis(self) -> int:
        return int(self.to_split_map.shape[0])

    @property
    def ngroups(self) -> int:
        return int(self.group_key.shape[0])

    @property
    def splitted_mol(self):
        if self._splitted_mol is None:
            raise ValueError("splitted_mol is not available")
        return self._splitted_mol

    @property
    def angs_no_pad(self):
        return self.angs[~self.pad_id]

    @property
    def ao_loc(self) -> np.ndarray:
        """Kernel-side cartesian AO offsets, (nbasis+1,); pads have zero width."""
        if "ao_loc" not in self._cache:
            dims = (self.angs + 1) * (self.angs + 2) // 2
            dims[self.pad_id] = 0
            loc = np.zeros(self.nbasis + 1, dtype=np.int32)
            np.cumsum(dims, out=loc[1:])
            self._cache["ao_loc"] = loc
        return self._cache["ao_loc"]

    @property
    def ao_loc_no_pad(self) -> np.ndarray:
        loc = self.ao_loc
        return np.concatenate([loc[:-1][~self.pad_id], loc[-1:]]).astype(np.int32)

    @property
    def nao(self) -> int:
        return int(self.ao_loc[-1])

    @property
    def to_decontracted_map(self) -> np.ndarray:
        out = np.full(self.nbasis, -1, dtype=np.int32)
        out[~self.pad_id] = self._split_to_decontracted[self.to_split_map[~self.pad_id]]
        return out

    def _mol_dec_ao_loc(self) -> np.ndarray:
        """AO offsets of the molecule's decontracted shells ((shell, contraction) pairs)."""
        bas = np.asarray(self._mol._bas)
        l = np.repeat(bas[:, ANG_OF], bas[:, NCTR_OF])
        dims = (l + 1) * (l + 2) // 2 if self._mol.cart else 2 * l + 1
        loc = np.zeros(len(dims) + 1, dtype=np.int32)
        np.cumsum(dims, out=loc[1:])
        return loc

    @property
    def mol_ao_loc(self) -> np.ndarray:
        """Molecule-side AO offset of every non-pad kernel shell (+ total at the end)."""
        loc = self._mol_dec_ao_loc()
        dec = self.to_decontracted_map[~self.pad_id]
        return np.concatenate([loc[dec], loc[-1:]]).astype(np.int32)

    @property
    def mol_ao_offset(self) -> np.ndarray:
        """(nbasis,) molecule-side AO offset per kernel shell, -1 for pads (engine input)."""
        loc = self._mol_dec_ao_loc()
        dec = self.to_decontracted_map
        return np.where(dec >= 0, loc[np.maximum(dec, 0)], -1).astype(np.int32)

    @property
    def shell_atom(self) -> np.ndarray:
        """(nbasis,) atom of each kernel-side shell, -1 for pads; split and decontracted shells map to
        the atom of their parent shell."""
        out = np.full(self.nbasis, -1, dtype=np.int32)
        out[~self.pad_id] = np.asarray(self.splitted_mol._bas)[self.to_split_map[~self.pad_id], ATOM_OF]
        return out

    @property
    def mol_nao(self) -> int:
        return int(self._mol_dec_ao_loc()[-1])

    @property
    def basis_data_fp64(self) -> dict:
        """Packed records, as the reference kernels take them (basis.py:326-371)."""
        if "packed" not in self._cache:
            packed = np.zeros((self.nbasis, BASIS_STRIDE), dtype=np.float64)
            packed[:, :3] = self.coords[:, :3]
            packed[:, 3] = self.ao_loc[:-1]
            packed[:, 4:] = self.ce
            self._cache["packed"] = {"coords": packed[:, :4].copy(), "ce": self.ce.astype(np.float64),
                                     "ao_loc": self.ao_loc.astype(np.float64), "packed": packed}
        return self._cache["packed"]

    # ------------------------------------------------------------------ engine plumbing
    def engine(self, devices=None):
        """The CUDA engine bound to this layout (created on first use, one per layout)."""
        key = ("engine", tuple(devices) if devices else None)
        if key not in self._cache:
            from ..backend.engine import JKEngine
            self._cache[key] = JKEngine(self, devices=devices)
        return self._cache[key]

    def q_matrix(self, omega=0.0):
        """log-Schwarz matrix (nbasis, nbasis) float32 on the device, cached per omega.
        The reference obtains it from libcint on the CPU (basis.py:218-243, 840-867); here it
        is evaluated by the engine on the GPU with the same definition."""
        return self.engine().q_matrix(0.0 if omega is None else float(omega))

    def dm_from_mol(self, mat):
        return self.engine().dm_from_mol(mat)

    def dm_to_mol(self, mat):
        return self.engine().dm_to_mol(mat)


def compute_q_matrix(layout_or_mol, omega=0.0):
    """Reference: basis.py:840-867 (libcint).  Device evaluation through the engine; accepts a
    BasisLayout (preferred) or a molecule."""
    layout = layout_or_mol if isinstance(layout_or_mol, BasisLayout) else BasisLayout.from_mol(layout_or_mol)
    return layout.q_matrix(omega)
