"""CPU checks of the J/K energy gradient oracle (tests/grad_oracle.c) and of BasisLayout.shell_atom.

The oracle's gradient is checked against 4-point finite differences of the oracle's own E_jk
(built from its already pinned get_jk) at displaced geometries, one coordinate at a time, and for
translational invariance, which is a real check because the oracle evaluates all four centres.
"""
import numpy as np
import pytest

from joltqc_b200.chem.mole import M
from joltqc_b200.pyscf.basis import BasisLayout
from tests import grad_oracle
from tests.common import H2O, random_dm

H = 1e-3           # Bohr; the 4-point difference is stable to ~1e-12 relative for h in [5e-4, 2e-3]
NO_SCREEN = 1e-30  # cutoff for the finite-difference comparisons (no quartet enters or leaves the screen)

CH4 = "C 0 0 0; H 0 0 1.09; H 1.03 0 -0.36; H -0.51 0.89 -0.36; H -0.51 -0.89 -0.36"


def _geometry(atom):
    mol = M(atom=atom, basis="sto-3g")
    return [mol.atom_symbol(a) for a in range(mol.natm)], mol.atom_coords()


def _layout(symbols, coords, basis, cart):
    atom = [(s, tuple(c)) for s, c in zip(symbols, coords)]
    mol = M(atom=atom, basis=basis, cart=cart, unit="B")
    return mol, BasisLayout.from_mol(mol, alignment=4)


def energy_jk(lay, dm, j_factor, k_factor, omega, cutoff=NO_SCREEN):
    """E_jk = (j/2) tr(D J) - (k/4) tr(D K) from the oracle's J/K build."""
    from oracle.oracle import OracleJK
    vj, vk = OracleJK(lay).get_jk(dm, 1, True, True, omega, cutoff)
    return 0.5 * j_factor * np.einsum("ij,ji", dm, vj) - 0.25 * k_factor * np.einsum("ij,ji", dm, vk)


def fd_gradient(symbols, coords, basis, cart, dm, j_factor, k_factor, omega, coords_to_check):
    out = {}
    for a, x in coords_to_check:
        f = {}
        for s in (-2, -1, 1, 2):
            c = coords.copy()
            c[a, x] += s * H
            f[s] = energy_jk(_layout(symbols, c, basis, cart)[1], dm, j_factor, k_factor, omega)
        out[a, x] = (-f[2] + 8 * f[1] - 8 * f[-1] + f[-2]) / (12 * H)
    return out


CASES = [
    # (id, atom, basis, cart, j_factor, k_factor, omega)
    ("h2o-svp-sph", H2O, "def2-svp", False, 1.0, 1.0, None),
    ("h2o-tzvpp-cart", H2O, "def2-tzvpp", True, 1.0, 1.0, None),
    ("h2o-spdfg", H2O, "test-spdfg", False, 1.0, 1.0, None),
    ("ch4-ccpvtz", CH4, "cc-pvtz", False, 1.0, 1.0, None),
    ("h2o-tzvpp-omega", H2O, "def2-tzvpp", False, 0.0, 0.6, 0.5),
    ("h2o-svp-j-only", H2O, "def2-svp", False, 1.0, 0.0, None),
    ("h2o-svp-k-only", H2O, "def2-svp", False, 0.0, 1.0, None),
]


def test_eri_twin_matches_pinned_eri_block():
    """the l <= 5 twin of eri_block used for the raised shells equals the pinned routine bitwise on random
    quartets of s to g shells (test-spdfg), Coulomb and long range"""
    from oracle.oracle import OracleJK
    mol = M(atom=H2O, basis="test-spdfg")
    lay = BasisLayout.from_mol(mol, alignment=4)
    orc = OracleJK(lay)
    real = np.nonzero(~lay.pad_id)[0]
    first = {}
    for s in real:                                # one shell per (l, atom)
        first.setdefault((int(lay.angs[s]), tuple(lay.coords[s, :3])), int(s))
    shells = sorted(first.values())
    assert max(int(lay.angs[s]) for s in shells) == 4
    rng = np.random.RandomState(0)
    for _ in range(60):
        i, j, k, l = (int(x) for x in rng.choice(shells, 4))
        for omega in (0.0, 0.5):
            ref = orc.eri_block(i, j, k, l, omega)
            assert np.array_equal(grad_oracle.eri_block(orc, i, j, k, l, omega), ref), (i, j, k, l, omega)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_gradient_vs_finite_differences(case):
    from oracle.oracle import OracleJK
    _, atom, basis, cart, jf, kf, omega = case
    symbols, coords = _geometry(atom)
    mol, lay = _layout(symbols, coords, basis, cart)
    dm = random_dm(mol.nao, 9) / mol.nao
    g, nq = grad_oracle.jk_energy_grad(OracleJK(lay), dm, jf, kf, omega, NO_SCREEN)
    assert g.shape == (mol.natm, 3) and nq > 0
    # every coordinate of the small molecules; for CH4/cc-pVTZ the carbon and one hydrogen
    atoms = range(mol.natm) if mol.natm <= 3 else (0, 1)
    fd = fd_gradient(symbols, coords, basis, cart, dm, jf, kf, omega, [(a, x) for a in atoms for x in range(3)])
    tol = 1e-9 * max(1.0, np.abs(g).max())
    err = max(abs(g[a, x] - v) for (a, x), v in fd.items())
    assert err < tol, (err, tol)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_gradient_translational_sum(case):
    from oracle.oracle import OracleJK
    _, atom, basis, cart, jf, kf, omega = case
    symbols, coords = _geometry(atom)
    mol, lay = _layout(symbols, coords, basis, cart)
    g, _ = grad_oracle.jk_energy_grad(OracleJK(lay), random_dm(mol.nao, 9) / mol.nao, jf, kf, omega)
    assert np.abs(g.sum(axis=0)).max() < 1e-10 * np.abs(g).max()


def test_oracle_gradient_screen_counts():
    """j-only and k-only screens keep subsets of the J+K screen's quartets"""
    from oracle.oracle import OracleJK
    mol = M(atom=H2O, basis="def2-svp")
    lay = BasisLayout.from_mol(mol, alignment=4)
    dm = random_dm(mol.nao, 3) * 1e-3
    orc = OracleJK(lay)
    n_jk = grad_oracle.jk_energy_grad(orc, dm, 1.0, 1.0, None, 1e-7)[1]
    n_j = grad_oracle.jk_energy_grad(orc, dm, 1.0, 0.0, None, 1e-7)[1]
    n_k = grad_oracle.jk_energy_grad(orc, dm, 0.0, 1.0, None, 1e-7)[1]
    n_all = grad_oracle.jk_energy_grad(orc, dm, 1.0, 1.0, None, 1e-30)[1]
    assert max(n_j, n_k) <= n_jk < n_all


def test_shell_atom_split_and_decontracted():
    """cc-pVTZ carbon has generally contracted s/p shells (decontracted into several kernel shells)
    and shells with more than three primitives (split): every piece maps to its parent's atom"""
    mol = M(atom=CH4, basis="cc-pvtz")
    lay = BasisLayout.from_mol(mol, alignment=4)
    sa = lay.shell_atom
    assert sa.shape == (lay.nbasis,) and sa.dtype == np.int32
    assert np.all(sa[lay.pad_id] == -1)
    assert np.all(sa[~lay.pad_id] >= 0) and np.all(sa[~lay.pad_id] < mol.natm)
    # coordinates of each kernel shell are its atom's coordinates
    xyz = mol.atom_coords()
    real = ~lay.pad_id
    assert np.allclose(lay.coords[real, :3], xyz[sa[real]])
    # per atom, the kernel shells cover exactly the molecule's AOs of that atom
    bas = np.asarray(mol._bas)
    mol_atom_of_ao = np.repeat(bas[:, 0], (2 * bas[:, 1] + 1) * bas[:, 3])   # spherical AOs: (2l+1) x nctr
    off = lay.mol_ao_offset
    for s in np.nonzero(real)[0]:
        assert mol_atom_of_ao[off[s]] == sa[s]
    # the carbon (atom 0) owns more kernel shells than molecular shells: split/decontracted pieces
    n_mol_c = int(np.sum(np.asarray(mol._bas)[:, 0] == 0))
    assert int(np.sum(sa == 0)) > n_mol_c
