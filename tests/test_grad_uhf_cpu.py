"""CPU checks of the spin-unrestricted J/K energy gradient oracle (grad_oracle_uhf.jk_energy_grad_uhf).

    E_U = (j/2) tr(Dt J[Dt]) - (k/2) [tr(Da K[Da]) + tr(Db K[Db])],   Dt = Da + Db

The oracle is checked against 4-point finite differences of E_U built from the pinned oracle's get_jk on
[Da, Db], against the three closed-shell oracle calls that compose the same gradient, against the
closed-shell oracle for Da = Db = D/2, and for translational invariance.  The two spin densities come
from different seeds, so the two K terms differ.
"""
import numpy as np
import pytest

from joltqc_b200.chem.mole import M
from joltqc_b200.pyscf.basis import BasisLayout
from tests import grad_oracle, grad_oracle_uhf
from tests.common import H2O, random_dm

H = 1e-3           # Bohr, as in test_grad_cpu.py
NO_SCREEN = 1e-30  # no quartet enters or leaves the screen between displaced geometries


def _geometry(atom):
    mol = M(atom=atom, basis="sto-3g")
    return [mol.atom_symbol(a) for a in range(mol.natm)], mol.atom_coords()


def _layout(symbols, coords, basis, cart=False):
    atom = [(s, tuple(c)) for s, c in zip(symbols, coords)]
    mol = M(atom=atom, basis=basis, cart=cart, unit="B")
    return mol, BasisLayout.from_mol(mol, alignment=4)


def _oracle(lay):
    from oracle.oracle import OracleJK
    return OracleJK(lay)


def spin_dms(nao):
    return np.stack([random_dm(nao, 9) / nao, random_dm(nao, 4) / nao])


def energy_uhf(lay, dm, j_factor, k_factor, omega, cutoff=NO_SCREEN):
    """E_U from the pinned oracle's J/K build on [Da, Db] (hermi = 1)."""
    vj, vk = _oracle(lay).get_jk(dm, 1, True, True, omega, cutoff)
    dt = dm[0] + dm[1]
    return (0.5 * j_factor * np.einsum("ij,ji", dt, vj[0] + vj[1])
            - 0.5 * k_factor * (np.einsum("ij,ji", dm[0], vk[0]) + np.einsum("ij,ji", dm[1], vk[1])))


CASES = [
    # (id, atom, basis, j_factor, k_factor, omega)
    ("h2o-svp", H2O, "def2-svp", 1.0, 1.0, None),
    ("h2o-spdfg", H2O, "test-spdfg", 1.0, 1.0, None),
    ("h2o-tzvpp-omega", H2O, "def2-tzvpp", 0.0, 0.6, 0.5),
    ("h2o-svp-j-only", H2O, "def2-svp", 1.0, 0.0, None),
    ("h2o-svp-k-only", H2O, "def2-svp", 0.0, 1.0, None),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_uhf_gradient_vs_finite_differences(case):
    _, atom, basis, jf, kf, omega = case
    symbols, coords = _geometry(atom)
    mol, lay = _layout(symbols, coords, basis)
    dm = spin_dms(mol.nao)
    g, nq = grad_oracle_uhf.jk_energy_grad_uhf(_oracle(lay), dm, jf, kf, omega, NO_SCREEN)
    assert g.shape == (mol.natm, 3) and nq > 0
    err = 0.0
    for a in range(mol.natm):
        for x in range(3):
            f = {}
            for s in (-2, -1, 1, 2):
                c = coords.copy()
                c[a, x] += s * H
                f[s] = energy_uhf(_layout(symbols, c, basis)[1], dm, jf, kf, omega)
            fd = (-f[2] + 8 * f[1] - 8 * f[-1] + f[-2]) / (12 * H)
            err = max(err, abs(g[a, x] - fd))
    tol = 1e-9 * max(1.0, np.abs(g).max())
    assert err < tol, (err, tol)


@pytest.mark.parametrize("omega", [None, 0.5])
def test_oracle_uhf_equals_three_closed_shell_calls(omega):
    """g_U(Da, Db; j, k) = g(Da + Db; j, 0) + g(Da; 0, 2k) + g(Db; 0, 2k)"""
    mol = M(atom=H2O, basis="def2-svp")
    lay = BasisLayout.from_mol(mol, alignment=4)
    orc = _oracle(lay)
    dm = spin_dms(mol.nao)
    jf, kf = 1.0, 0.7
    g, _ = grad_oracle_uhf.jk_energy_grad_uhf(orc, dm, jf, kf, omega, 1e-14)
    ref = (grad_oracle.jk_energy_grad(orc, dm[0] + dm[1], jf, 0.0, omega, 1e-14)[0]
           + grad_oracle.jk_energy_grad(orc, dm[0], 0.0, 2 * kf, omega, 1e-14)[0]
           + grad_oracle.jk_energy_grad(orc, dm[1], 0.0, 2 * kf, omega, 1e-14)[0])
    assert np.abs(g - ref).max() < 1e-10 * max(1.0, np.abs(ref).max())


def test_oracle_uhf_equal_spins_is_closed_shell():
    """Da = Db = D/2 gives the closed-shell gradient of D"""
    mol = M(atom=H2O, basis="def2-tzvpp")
    lay = BasisLayout.from_mol(mol, alignment=4)
    orc = _oracle(lay)
    d = random_dm(mol.nao, 9) / mol.nao
    g, _ = grad_oracle_uhf.jk_energy_grad_uhf(orc, np.stack([d / 2, d / 2]), 1.0, 1.0, None, 1e-14)
    ref, _ = grad_oracle.jk_energy_grad(orc, d, 1.0, 1.0, None, 1e-14)
    assert np.abs(g - ref).max() < 1e-10 * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_uhf_translational_sum(case):
    _, atom, basis, jf, kf, omega = case
    symbols, coords = _geometry(atom)
    mol, lay = _layout(symbols, coords, basis)
    g, _ = grad_oracle_uhf.jk_energy_grad_uhf(_oracle(lay), spin_dms(mol.nao), jf, kf, omega)
    assert np.abs(g.sum(axis=0)).max() < 1e-10 * np.abs(g).max()
