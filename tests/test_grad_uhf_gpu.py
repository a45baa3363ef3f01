"""GPU tests of the spin-unrestricted J/K energy gradient (jqc_jk_energy_grad_uhf /
joltqc_b200.pyscf.grad.generate_jk_energy_per_atom_uhf).

    E_U = (j/2) tr(Dt J[Dt]) - (k/2) [tr(Da K[Da]) + tr(Db K[Db])],   Dt = Da + Db

Evidence that does not rely on the new kernel's own arithmetic: the CPU oracle's unrestricted gradient
(tests/grad_oracle_uhf.c, checked in tests/test_grad_uhf_cpu.py), the closed-shell engine call it must reduce
to, and finite differences of E_U from the engine's validated get_jk on [Da, Db] at displaced geometries.
"""
import numpy as np
import pytest

from joltqc_b200.chem.mole import M
from joltqc_b200.pyscf.basis import BasisLayout
from tests import grad_oracle_uhf
from tests.common import H2O, benzene, random_dm

pytestmark = pytest.mark.gpu
TOL = 1e-10
H = 1e-3
CH4 = "C 0 0 0; H 0 0 1.09; H 1.03 0 -0.36; H -0.51 0.89 -0.36; H -0.51 -0.89 -0.36"


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device")
    return torch


def _layout(atom, basis, cart=False, unit="Angstrom"):
    mol = M(atom=atom, basis=basis, cart=cart, unit=unit)
    return mol, BasisLayout.from_mol(mol, alignment=4)


def _oracle(lay):
    from oracle.oracle import OracleJK
    return OracleJK(lay)


def spin_dms(nao, scale=None):
    s = 1.0 / nao if scale is None else scale
    return np.stack([random_dm(nao, 9) * s, random_dm(nao, 4) * s])


def _engine_grad(lay, dm, jf=1.0, kf=1.0, omega=None, cutoff=1e-13):
    from joltqc_b200.pyscf.grad import generate_jk_energy_per_atom_uhf
    return generate_jk_energy_per_atom_uhf(lay, cutoff)(dm, j_factor=jf, k_factor=kf, omega=omega).cpu().numpy()


def _energy_gpu(symbols, coords_bohr, basis, dm, jf, kf, omega, cutoff):
    """E_U from the engine's get_jk on [Da, Db] at the given geometry (Bohr)."""
    from joltqc_b200.pyscf.jk import generate_jk_kernel
    atom = [(s, tuple(c)) for s, c in zip(symbols, coords_bohr)]
    mol, lay = _layout(atom, basis, unit="B")
    vj, vk = generate_jk_kernel(lay, cutoff, cutoff)(mol, dm, hermi=1, omega=omega)
    vj, vk = vj.cpu().numpy(), vk.cpu().numpy()
    dt = dm[0] + dm[1]
    return (0.5 * jf * np.einsum("ij,ji", dt, vj[0] + vj[1])
            - 0.5 * kf * (np.einsum("ij,ji", dm[0], vk[0]) + np.einsum("ij,ji", dm[1], vk[1])))


def _symbols_coords(mol):
    return [mol.atom_symbol(a) for a in range(mol.natm)], mol.atom_coords()


CASES = [
    # (id, atom, basis, cart, j_factor, k_factor, omega): the cases of test_grad_gpu.py
    ("h2o-svp-sph", H2O, "def2-svp", False, 1.0, 1.0, None),
    ("h2o-tzvpp-cart", H2O, "def2-tzvpp", True, 1.0, 1.0, None),
    ("h2o-spdfg", H2O, "test-spdfg", False, 1.0, 1.0, None),
    ("h2o-spdfg-cart", H2O, "test-spdfg", True, 1.0, 1.0, None),
    ("ch4-ccpvtz", CH4, "cc-pvtz", False, 1.0, 1.0, None),
    ("h2o-tzvpp-omega", H2O, "def2-tzvpp", False, 0.0, 0.6, 0.5),
    ("h2o-svp-j-only", H2O, "def2-svp", False, 1.0, 0.0, None),
    ("h2o-svp-k-only", H2O, "def2-svp", False, 0.0, 1.0, None),
    ("benzene-ccpvtz", benzene(), "cc-pvtz", False, 1.0, 1.0, None),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_engine_matches_oracle(torch_cuda, case):
    _, atom, basis, cart, jf, kf, omega = case
    mol, lay = _layout(atom, basis, cart=cart)
    dm = spin_dms(mol.nao)
    g = _engine_grad(lay, dm, jf, kf, omega)
    ref, _ = grad_oracle_uhf.jk_energy_grad_uhf(_oracle(lay), dm, jf, kf, omega)
    assert g.shape == (mol.natm, 3)
    err = np.abs(g - ref).max()
    assert err < TOL * max(1.0, np.abs(ref).max()), (err, np.abs(ref).max())


def test_convenience_function(torch_cuda):
    from joltqc_b200.pyscf.grad import jk_energy_per_atom_uhf
    mol, lay = _layout(H2O, "def2-svp")
    dm = spin_dms(mol.nao)
    g = jk_energy_per_atom_uhf(mol, dm, 1.0, 0.25).cpu().numpy()
    ref, _ = grad_oracle_uhf.jk_energy_grad_uhf(_oracle(lay), dm, 1.0, 0.25)
    assert np.abs(g - ref).max() < TOL * max(1.0, np.abs(ref).max())


def test_loose_cutoff_same_quartet_set(torch_cuda):
    """with a loose threshold many quartets are dropped; the engine must drop the same ones"""
    mol, lay = _layout(benzene(), "def2-svp")
    dm = spin_dms(mol.nao, 1e-3)
    eng = lay.engine()
    counts = {}
    for jf, kf in ((1.0, 1.0), (1.0, 0.0), (0.0, 1.0)):
        g = eng.jk_energy_grad_uhf(dm, lay.shell_atom, mol.natm, jf, kf, None, 1e-7, count=True).cpu().numpy()
        ref, nq = grad_oracle_uhf.jk_energy_grad_uhf(_oracle(lay), dm, jf, kf, None, 1e-7)
        assert eng.last_grad_quartets == nq, (jf, kf, eng.last_grad_quartets, nq)
        assert np.abs(g - ref).max() < 1e-12 * max(1.0, np.abs(ref).max())
        counts[jf, kf] = nq
    eng.jk_energy_grad_uhf(dm, lay.shell_atom, mol.natm, 1.0, 1.0, None, 1e-13, count=True)
    assert eng.last_grad_quartets > counts[1.0, 1.0]


@pytest.mark.parametrize("omega", [None, 0.5])
def test_equal_spins_is_closed_shell(torch_cuda, omega):
    """Da = Db = D/2 reproduces jk_energy_grad(D)"""
    mol, lay = _layout(H2O, "def2-tzvpp")
    d = random_dm(mol.nao, 9) / mol.nao
    eng = lay.engine()
    g = eng.jk_energy_grad_uhf(np.stack([d / 2, d / 2]), lay.shell_atom, mol.natm, 1.0, 0.8, omega, 1e-14)
    ref = eng.jk_energy_grad(d, lay.shell_atom, mol.natm, 1.0, 0.8, omega, 1e-14)
    g, ref = g.cpu().numpy(), ref.cpu().numpy()
    assert np.abs(g - ref).max() < TOL * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("omega", [None, 0.5])
def test_fused_equals_three_closed_shell_calls(torch_cuda, omega):
    """g_U(Da, Db; j, k) = g(Da + Db; j, 0) + g(Da; 0, 2k) + g(Db; 0, 2k), all on the engine"""
    mol, lay = _layout(H2O, "def2-tzvpp")
    dm = spin_dms(mol.nao)
    eng = lay.engine()
    sa, natm = lay.shell_atom, mol.natm
    jf, kf = 1.0, 0.7
    g = eng.jk_energy_grad_uhf(dm, sa, natm, jf, kf, omega, 1e-14).cpu().numpy()
    ref = (eng.jk_energy_grad(dm[0] + dm[1], sa, natm, jf, 0.0, omega, 1e-14)
           + eng.jk_energy_grad(dm[0], sa, natm, 0.0, 2 * kf, omega, 1e-14)
           + eng.jk_energy_grad(dm[1], sa, natm, 0.0, 2 * kf, omega, 1e-14)).cpu().numpy()
    assert np.abs(g - ref).max() < TOL * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("omega", [None, 0.5])
def test_finite_differences_of_engine_get_jk(torch_cuda, omega):
    """H2O/def2-TZVPP: every coordinate against a 4-point difference of E_U from four get_jk builds"""
    mol, lay = _layout(H2O, "def2-tzvpp")
    symbols, coords = _symbols_coords(mol)
    dm = spin_dms(mol.nao)
    g = _engine_grad(lay, dm, 1.0, 1.0, omega, cutoff=1e-14)
    err = 0.0
    for a in range(mol.natm):
        for x in range(3):
            f = {}
            for s in (-2, -1, 1, 2):
                c = coords.copy()
                c[a, x] += s * H
                f[s] = _energy_gpu(symbols, c, "def2-tzvpp", dm, 1.0, 1.0, omega, 1e-14)
            fd = (-f[2] + 8 * f[1] - 8 * f[-1] + f[-2]) / (12 * H)
            err = max(err, abs(g[a, x] - fd))
    scale = max(1.0, np.abs(g).max())
    print(f"\nH2O/def2-TZVPP UHF omega={omega}: max|g - fd| = {err:.3e} (max|g| = {np.abs(g).max():.3f})")
    assert err < 1e-7 * scale, (err, scale)


def test_directional_finite_difference_benzene(torch_cuda):
    """benzene/cc-pVTZ: g.u for one random unit displacement u of all atoms against four get_jk builds"""
    mol, lay = _layout(benzene(), "cc-pvtz")
    symbols, coords = _symbols_coords(mol)
    dm = spin_dms(mol.nao)
    g = _engine_grad(lay, dm, 1.0, 1.0, None, cutoff=1e-14)
    u = np.random.RandomState(5).randn(*coords.shape)
    u /= np.linalg.norm(u)
    f = {s: _energy_gpu(symbols, coords + s * H * u, "cc-pvtz", dm, 1.0, 1.0, None, 1e-14) for s in (-2, -1, 1, 2)}
    fd = (-f[2] + 8 * f[1] - 8 * f[-1] + f[-2]) / (12 * H)
    gu = float(np.sum(g * u))
    print(f"\nbenzene/cc-pVTZ UHF: g.u = {gu:.12f}, 4-point fd = {fd:.12f}, diff = {gu - fd:.3e}")
    assert abs(gu - fd) < 1e-7 * max(1.0, np.abs(g).max())


def test_shards_sum_to_full_gradient(torch_cuda):
    """ranks 0..2 of a world of 3 on one GPU: partial gradients sum to the full one, every quartet once"""
    from joltqc_b200.backend.engine import JKEngine
    mol, lay = _layout(benzene(), "def2-svp")
    dm = spin_dms(mol.nao)
    full_eng = lay.engine()
    full = full_eng.jk_energy_grad_uhf(dm, lay.shell_atom, mol.natm, count=True)
    n_full = full_eng.last_grad_quartets
    eng = JKEngine(lay)
    total, n = None, 0
    for rank in range(3):
        eng.set_shard(rank, 3)
        part = eng.jk_energy_grad_uhf(dm, lay.shell_atom, mol.natm, count=True)
        n += eng.last_grad_quartets
        total = part.clone() if total is None else total + part
    assert n == n_full
    assert (total - full).abs().max().item() < 1e-12 * full.abs().max().item()


def test_jk_state_untouched(torch_cuda):
    """build_partial([Da, Db]) -> unrestricted gradient -> finalize: the [J || K] buffer is bitwise unchanged,
    the accounting of the J/K build still reads the same and finalize still gives the oracle's J and K"""
    import torch
    mol, lay = _layout(H2O, "def2-tzvpp")
    dm = spin_dms(mol.nao)
    eng = lay.engine()
    buf = eng.build_partial(dm, hermi=1)
    torch.cuda.synchronize()
    before = buf.clone()
    counts_before = eng.last_stats()[0]
    g = eng.jk_energy_grad_uhf(dm, lay.shell_atom, mol.natm, count=True)
    torch.cuda.synchronize()
    assert torch.equal(buf, before)
    assert np.array_equal(eng.last_stats()[0], counts_before)
    vj, vk = eng.finalize()
    rj, rk = _oracle(lay).get_jk(dm, 1)
    assert np.abs(vj.cpu().numpy() - rj).max() < TOL * max(1.0, np.abs(rj).max())
    assert np.abs(vk.cpu().numpy() - rk).max() < TOL * max(1.0, np.abs(rk).max())
    assert g.shape == (mol.natm, 3) and eng.last_grad_quartets > 0


def test_rejected_inputs(torch_cuda):
    from joltqc_b200.backend.lib import JQCError
    from joltqc_b200.pyscf.grad import generate_jk_energy_per_atom_uhf
    mol, lay = _layout(H2O, "def2-svp")
    grad = generate_jk_energy_per_atom_uhf(lay)
    dm = spin_dms(mol.nao)
    with pytest.raises(AssertionError):
        grad(dm, omega=-0.3)
    with pytest.raises(ValueError):
        grad(dm[0])                                  # one density
    with pytest.raises(ValueError):
        grad(np.stack([dm[0], dm[1], dm[0]]))        # three densities
    with pytest.raises(ValueError):
        grad(dm[:, :-1, :-1])                        # wrong nao
    for s in range(2):
        bad = dm.copy()
        bad[s] = random_dm(mol.nao, 9, symmetric=False)
        with pytest.raises(ValueError):
            grad(bad)
    with pytest.raises(ValueError):
        grad(dm, j_factor=0.0, k_factor=0.0)
    # the C ABI's own checks
    eng = lay.engine()
    sa = lay.shell_atom
    with pytest.raises(ValueError):
        eng.jk_energy_grad_uhf(dm[0], sa, mol.natm)
    with pytest.raises(JQCError):
        eng.jk_energy_grad_uhf(dm, sa, mol.natm, 0.0, 0.0)
    with pytest.raises(JQCError):
        eng.jk_energy_grad_uhf(dm, sa, mol.natm, omega=-0.3)
    with pytest.raises(JQCError):
        eng.jk_energy_grad_uhf(dm, sa, mol.natm, cutoff=0.0)
    with pytest.raises(JQCError):
        eng.jk_energy_grad_uhf(dm, sa, 0)
    bad = sa.copy()
    bad[0] = mol.natm
    with pytest.raises(JQCError):
        eng.jk_energy_grad_uhf(dm, bad, mol.natm)
