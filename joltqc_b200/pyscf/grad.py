"""Nuclear gradient of the J/K energy, backed by the CUDA engine.

For a symmetric density ``D`` in the molecule's AO basis,

    E_jk(R) = (j_factor / 2) tr(D J[D]) - (k_factor / 4) tr(D K[D])

with ``J, K = get_jk(mol, D, hermi=1, omega=omega)``.  ``D`` is held fixed and the basis functions
move with their atoms; the result is ``dE_jk / dR`` as an ``(natm, 3)`` array in Hartree/Bohr on the
engine's device.  This is the two-electron part of an SCF gradient evaluated with the energy-weighted
density left to the caller:

* RHF: ``j_factor = k_factor = 1``;
* hybrid RKS: ``k_factor = hyb``;
* range-separated hybrid: a second call with ``omega = w``, ``j_factor = 0`` and
  ``k_factor = alpha - hyb``, as ``rks.py`` combines ``get_jk`` and ``get_k(omega=)``.

For the two spin densities ``Da, Db`` of an unrestricted calculation (the ``(2, nao, nao)`` array of
``make_rdm1()``) and ``Dt = Da + Db``, ``generate_jk_energy_per_atom_uhf`` gives the gradient of

    E_U(R) = (j_factor / 2) tr(Dt J[Dt]) - (k_factor / 2) [tr(Da K[Da]) + tr(Db K[Db])]

with ``J, K = get_jk(mol, [Da, Db], hermi=1, omega=omega)``, in one pass over the derivative integrals.
The factor conventions are the same (UHF: ``j_factor = k_factor = 1``; UKS hybrid: ``k_factor = hyb``;
long-range part: a second call with ``omega``, ``j_factor = 0``, ``k_factor = alpha - hyb``).  With
``Da = Db = D / 2`` it equals the closed-shell gradient of ``D``.

Symmetric densities, ``hermi = 1`` and FP64 only.  Like ``jk.py`` this module holds no arithmetic.
"""
from ..constants import TILE
from .basis import BasisLayout

__all__ = ["generate_jk_energy_per_atom", "jk_energy_per_atom", "generate_jk_energy_per_atom_uhf",
           "jk_energy_per_atom_uhf"]


def _check_dm(d, nao):
    if d.ndim != 2 or d.shape[0] != nao or d.shape[1] != nao:
        raise ValueError(f"dm has shape {tuple(d.shape)}, the molecule has {nao} AOs (one 2-D density)")
    scale = d.abs().max().item()
    if (d - d.T).abs().max().item() > 1e-12 * scale:
        raise ValueError("dm is not symmetric: the J/K energy gradient needs a hermi = 1 density")


def generate_jk_energy_per_atom(basis_layout: BasisLayout, cutoff=1e-13):
    """Returns ``grad(dm, j_factor=1.0, k_factor=1.0, omega=None) -> (natm, 3)``.  A CuPy ``dm`` gets a
    CuPy result, anything else a torch tensor on the engine's device."""
    assert basis_layout.alignment % TILE == 0, "the J/K layout must be padded to TILE"
    engine = basis_layout.engine()
    shell_atom = basis_layout.shell_atom
    natm = int(basis_layout._mol.natm)

    def grad(dm, j_factor=1.0, k_factor=1.0, omega=None):
        if omega is not None:
            assert omega >= 0.0, "short ranged J/K not supported"
        if j_factor == 0 and k_factor == 0:
            raise ValueError("j_factor and k_factor are both zero")
        d = engine._dev(dm)
        _check_dm(d, engine.mol_nao)
        g = engine.jk_energy_grad(d, shell_atom, natm, j_factor=j_factor, k_factor=k_factor, omega=omega,
                                  cutoff=cutoff)
        if type(dm).__module__.split(".")[0] == "cupy":
            import cupy as cp
            g = cp.from_dlpack(g)
        return g

    grad.engine = engine
    return grad


def jk_energy_per_atom(mol, dm, j_factor=1.0, k_factor=1.0, omega=None, cutoff=1e-13):
    """Convenience form, like ``jk.get_jk(mol, ...)``: builds the layout of ``mol`` and evaluates once."""
    layout = BasisLayout.from_mol(mol, alignment=TILE)
    return generate_jk_energy_per_atom(layout, cutoff)(dm, j_factor=j_factor, k_factor=k_factor, omega=omega)


def generate_jk_energy_per_atom_uhf(basis_layout: BasisLayout, cutoff=1e-13):
    """Returns ``grad(dm, j_factor=1.0, k_factor=1.0, omega=None) -> (natm, 3)`` for the spin densities
    ``dm = [Da, Db]`` of shape ``(2, nao, nao)``.  A CuPy ``dm`` gets a CuPy result, anything else a torch
    tensor on the engine's device."""
    assert basis_layout.alignment % TILE == 0, "the J/K layout must be padded to TILE"
    engine = basis_layout.engine()
    shell_atom = basis_layout.shell_atom
    natm = int(basis_layout._mol.natm)

    def grad(dm, j_factor=1.0, k_factor=1.0, omega=None):
        if omega is not None:
            assert omega >= 0.0, "short ranged J/K not supported"
        if j_factor == 0 and k_factor == 0:
            raise ValueError("j_factor and k_factor are both zero")
        d = engine._dev(dm)
        if d.ndim != 3 or d.shape[0] != 2:
            raise ValueError(f"dm has shape {tuple(d.shape)}: the unrestricted gradient takes (2, nao, nao) "
                             "spin densities [Da, Db]")
        for s in range(2):
            _check_dm(d[s], engine.mol_nao)
        g = engine.jk_energy_grad_uhf(d, shell_atom, natm, j_factor=j_factor, k_factor=k_factor, omega=omega,
                                      cutoff=cutoff)
        if type(dm).__module__.split(".")[0] == "cupy":
            import cupy as cp
            g = cp.from_dlpack(g)
        return g

    grad.engine = engine
    return grad


def jk_energy_per_atom_uhf(mol, dm, j_factor=1.0, k_factor=1.0, omega=None, cutoff=1e-13):
    """Convenience form of ``generate_jk_energy_per_atom_uhf``: builds the layout of ``mol`` and evaluates once."""
    layout = BasisLayout.from_mol(mol, alignment=TILE)
    return generate_jk_energy_per_atom_uhf(layout, cutoff)(dm, j_factor=j_factor, k_factor=k_factor, omega=omega)
