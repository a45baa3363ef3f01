"""Device time of the J/K energy gradient (jqc_jk_energy_grad) next to the J/K build on the same density.

For each workload one JSON line: seconds per gradient build (CUDA events, warmed up), quartets evaluated,
seconds per J/K build in the same run and the ratio, the GPU's name, power limit and SM clock read in
the same run, and (for the workloads named by --fd) a directional finite-difference check: g.u for one
random unit displacement u of all atoms against a 4-point difference of
E_jk = 1/2 tr(D J) - 1/4 tr(D K) from four get_jk builds at displaced geometries.

    python tools/grad_bench.py [--steps 3] [--warmup 1] [--fd taxol-svp]

With --uhf the spin-unrestricted gradient (jqc_jk_energy_grad_uhf) is timed instead, on the spin
densities Da = D/2 + S, Db = D/2 - S, where D is the decaying model density and S a seeded symmetric
matrix with the same exp(-0.6 r) envelope, scaled by 0.1.  Each line then holds the seconds per fused
unrestricted gradient, per composition of the same result from three closed-shell calls
(g(Dt; j, 0) + g(Da; 0, 2k) + g(Db; 0, 2k)), per closed-shell gradient of Dt and per J/K build of Dt, all
from the same run; the quartet counts; max |fused - composed|; and the directional finite-difference
check on E_U = 1/2 tr(Dt J[Dt]) - 1/2 [tr(Da K[Da]) + tr(Db K[Db])] from four get_jk builds on [Da, Db].

Workloads and the decaying model density are bench.py's (bench.build_mol, bench.make_dm).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402

H = 1e-3        # Bohr
CUTOFF = 1e-13  # timed builds
FD_CUTOFF = 1e-14


def gpu_info(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_clock_mhz": float(out[2]), "sm_max_mhz": float(out[3])}
    except Exception as exc:  # the timing itself does not need nvidia-smi
        import torch
        return {"gpu": torch.cuda.get_device_name(index), "power_limit_w": None, "sm_clock_mhz": None,
                "nvidia_smi": repr(exc)}


def progress(msg):
    print(msg, file=sys.stderr, flush=True)


def time_grad(eng, lay, natm, dm_dev, warmup, steps):
    """Seconds per gradient build and the quartet count (read during the warm-up builds)."""
    import torch
    for _ in range(max(1, warmup)):
        eng.jk_energy_grad(dm_dev, lay.shell_atom, natm, cutoff=CUTOFF, count=True)
        progress(f"  warm-up gradient build: {eng.last_grad_quartets} quartets")
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        g = eng.jk_energy_grad(dm_dev, lay.shell_atom, natm, cutoff=CUTOFF)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / steps, g, eng.last_grad_quartets


def energy_jk(mol, coords, dm_dev):
    """E_jk at displaced coordinates (Bohr) from the engine's get_jk."""
    import torch
    from joltqc_b200.chem.mole import M
    from joltqc_b200.pyscf.basis import BasisLayout
    atom = [(mol.atom_symbol(a), tuple(c)) for a, c in enumerate(coords)]
    m = M(atom=atom, basis=mol.basis, cart=mol.cart, unit="B")
    lay = BasisLayout.from_mol(m, alignment=4)
    vj, vk = lay.engine().get_jk(dm_dev, hermi=1, cutoff_fp64=FD_CUTOFF, cutoff_fp32=FD_CUTOFF)
    e = 0.5 * torch.sum(dm_dev * vj).item() - 0.25 * torch.sum(dm_dev * vk).item()
    lay._cache.clear()
    torch.cuda.empty_cache()
    return e


def directional_fd(mol, lay, dm_dev):
    g = lay.engine().jk_energy_grad(dm_dev, lay.shell_atom, mol.natm, cutoff=FD_CUTOFF).cpu().numpy()
    coords = mol.atom_coords()
    u = np.random.RandomState(11).randn(*coords.shape)
    u /= np.linalg.norm(u)
    f = {}
    for s in (-2, -1, 1, 2):
        f[s] = energy_jk(mol, coords + s * H * u, dm_dev)
        progress(f"  E_jk at displacement {s} h: {f[s]:.12f}")
    fd = (-f[2] + 8 * f[1] - 8 * f[-1] + f[-2]) / (12 * H)
    gu = float(np.sum(g * u))
    return {"g_dot_u": gu, "fd_4point": fd, "abs_err": abs(gu - fd), "rel_err": abs(gu - fd) / max(abs(gu), 1e-300),
            "h_bohr": H, "cutoff": FD_CUTOFF, "max_abs_g": float(np.abs(g).max())}


def spin_dms(mol):
    """Da = D/2 + S, Db = D/2 - S (see the module docstring)."""
    d = bench.make_dm(mol, "decay")
    rng = np.random.RandomState(13)
    atom_of = np.repeat(mol._bas[:, 0], np.diff(mol.ao_loc))
    xyz = mol.atom_coords()[atom_of]
    dist = np.linalg.norm(xyz[:, None, :] - xyz[None, :, :], axis=-1)
    r = rng.randn(mol.nao, mol.nao)
    s = 0.1 * 0.5 * (r + r.T) * np.exp(-0.6 * dist)
    return np.stack([0.5 * d + s, 0.5 * d - s])


def time_calls(fn, warmup, steps):
    """Seconds per call of fn() (CUDA events after warm-up) and its last result."""
    import torch
    for _ in range(max(1, warmup)):
        out = fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / steps, out


def energy_uhf(mol, coords, dm_dev):
    """E_U at displaced coordinates (Bohr) from the engine's get_jk on [Da, Db]."""
    import torch
    from joltqc_b200.chem.mole import M
    from joltqc_b200.pyscf.basis import BasisLayout
    atom = [(mol.atom_symbol(a), tuple(c)) for a, c in enumerate(coords)]
    m = M(atom=atom, basis=mol.basis, cart=mol.cart, unit="B")
    lay = BasisLayout.from_mol(m, alignment=4)
    vj, vk = lay.engine().get_jk(dm_dev, hermi=1, cutoff_fp64=FD_CUTOFF, cutoff_fp32=FD_CUTOFF)
    dt = dm_dev[0] + dm_dev[1]
    e = 0.5 * torch.sum(dt * (vj[0] + vj[1])).item() - 0.5 * torch.sum(dm_dev * vk).item()
    lay._cache.clear()
    torch.cuda.empty_cache()
    return e


def directional_fd_uhf(mol, lay, dm_dev):
    g = lay.engine().jk_energy_grad_uhf(dm_dev, lay.shell_atom, mol.natm, cutoff=FD_CUTOFF).cpu().numpy()
    coords = mol.atom_coords()
    u = np.random.RandomState(11).randn(*coords.shape)
    u /= np.linalg.norm(u)
    f = {}
    for s in (-2, -1, 1, 2):
        f[s] = energy_uhf(mol, coords + s * H * u, dm_dev)
        progress(f"  E_U at displacement {s} h: {f[s]:.12f}")
    fd = (-f[2] + 8 * f[1] - 8 * f[-1] + f[-2]) / (12 * H)
    gu = float(np.sum(g * u))
    return {"g_dot_u": gu, "fd_4point": fd, "abs_err": abs(gu - fd), "rel_err": abs(gu - fd) / max(abs(gu), 1e-300),
            "h_bohr": H, "cutoff": FD_CUTOFF, "max_abs_g": float(np.abs(g).max())}


def run_uhf(wl, mol, label, lay, eng, dev, args, fd_set):
    import torch
    dm_dev = torch.as_tensor(spin_dms(mol), device=dev)
    dt_dev = dm_dev[0] + dm_dev[1]
    sa, natm, steps = lay.shell_atom, mol.natm, max(3, args.steps)
    sampler = bench.ClockSampler(dev.index)
    sampler.start()
    progress(f"{wl}: nao {mol.nao}, unrestricted")

    def fused():
        return eng.jk_energy_grad_uhf(dm_dev, sa, natm, cutoff=CUTOFF)

    def composed():
        return (eng.jk_energy_grad(dt_dev, sa, natm, 1.0, 0.0, cutoff=CUTOFF)
                + eng.jk_energy_grad(dm_dev[0], sa, natm, 0.0, 2.0, cutoff=CUTOFF)
                + eng.jk_energy_grad(dm_dev[1], sa, natm, 0.0, 2.0, cutoff=CUTOFF))

    def closed():
        return eng.jk_energy_grad(dt_dev, sa, natm, cutoff=CUTOFF)

    fused_s, g = time_calls(fused, args.warmup, steps)
    progress(f"  fused unrestricted gradient: {fused_s:.3f} s")
    composed_s, g3 = time_calls(composed, args.warmup, steps)
    progress(f"  three closed-shell calls: {composed_s:.3f} s")
    closed_s, _ = time_calls(closed, args.warmup, steps)
    progress(f"  closed-shell gradient of Dt: {closed_s:.3f} s")
    jk_s = bench.time_builds(eng, dt_dev, args.warmup, steps) * 1e-3
    progress(f"  J/K of Dt: {jk_s:.3f} s")
    clocks = sampler.stop()
    # quartet counts, outside the timed windows
    eng.jk_energy_grad_uhf(dm_dev, sa, natm, cutoff=CUTOFF, count=True)
    n_fused = eng.last_grad_quartets
    n_comp = 0
    for d, jf, kf in ((dt_dev, 1.0, 0.0), (dm_dev[0], 0.0, 2.0), (dm_dev[1], 0.0, 2.0)):
        eng.jk_energy_grad(d, sa, natm, jf, kf, cutoff=CUTOFF, count=True)
        n_comp += eng.last_grad_quartets
    eng.jk_energy_grad(dt_dev, sa, natm, cutoff=CUTOFF, count=True)
    n_closed = eng.last_grad_quartets
    jk_counts, _, _ = eng.last_stats()
    max_g = float(g.abs().max().item())
    out = {"workload": wl, "label": label, "nao": mol.nao, "natm": mol.natm, "dm": "decay +- 0.1 S (unrestricted)",
           "cutoff": CUTOFF, "steps": steps,
           "uhf_s_per_grad": fused_s, "three_call_s": composed_s, "closed_shell_grad_dt_s": closed_s,
           "jk_dt_s_per_build": jk_s, "uhf_over_closed_shell": fused_s / closed_s,
           "three_call_over_uhf": composed_s / fused_s, "uhf_over_jk": fused_s / jk_s,
           "uhf_quartets": n_fused, "three_call_quartets": n_comp, "closed_shell_quartets": n_closed,
           "jk_quartets": int(jk_counts.sum()), "max_abs_fused_minus_composed": float((g - g3).abs().max().item()),
           "max_abs_g": max_g, "translational_sum": float(g.sum(dim=0).abs().max().item()),
           "sampled_sm_mhz": clocks.get("sm_mhz"), "clock_reasons": clocks.get("reasons")}
    out["fused_matches_composed"] = out["max_abs_fused_minus_composed"] < 1e-10 * max(1.0, max_g)
    out.update(gpu_info(dev.index))
    if wl in fd_set:
        out["directional_fd"] = directional_fd_uhf(mol, lay, dm_dev)
        out["directional_fd"]["passed"] = out["directional_fd"]["abs_err"] < 1e-7 * max(1.0, max_g)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="taxol-svp,valinomycin-tzvp")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--fd", default="taxol-svp", help="comma-separated workloads that also run the finite-difference check")
    ap.add_argument("--uhf", action="store_true", help="time the spin-unrestricted gradient against three closed-shell calls")
    args = ap.parse_args()
    import torch
    from joltqc_b200.pyscf.basis import BasisLayout
    dev = torch.device("cuda", torch.cuda.current_device())
    fd_set = set(filter(None, args.fd.split(",")))
    for wl in args.workloads.split(","):
        mol, label = bench.build_mol(wl)
        lay = BasisLayout.from_mol(mol, alignment=4)
        eng = lay.engine()
        eng.q_matrix(0.0)
        if args.uhf:
            print(json.dumps(run_uhf(wl, mol, label, lay, eng, dev, args, fd_set)), flush=True)
            lay._cache.clear()
            del eng
            torch.cuda.empty_cache()
            continue
        dm_dev = torch.as_tensor(bench.make_dm(mol, "decay"), device=dev)
        sampler = bench.ClockSampler(dev.index)
        sampler.start()
        progress(f"{wl}: nao {mol.nao}")
        grad_s, g, grad_quartets = time_grad(eng, lay, mol.natm, dm_dev, args.warmup, max(3, args.steps))
        progress(f"  gradient: {grad_s:.3f} s per build")
        jk_s = bench.time_builds(eng, dm_dev, args.warmup, max(3, args.steps)) * 1e-3
        progress(f"  J/K: {jk_s:.3f} s per build")
        clocks = sampler.stop()
        jk_counts, _, _ = eng.last_stats()
        out = {"workload": wl, "label": label, "nao": mol.nao, "natm": mol.natm, "dm": "decay", "cutoff": CUTOFF,
               "grad_s_per_build": grad_s, "grad_quartets": grad_quartets, "steps": max(3, args.steps),
               "jk_s_per_build": jk_s, "jk_quartets": int(jk_counts.sum()), "grad_over_jk": grad_s / jk_s,
               "translational_sum": float(g.sum(dim=0).abs().max().item()), "max_abs_g": float(g.abs().max().item()),
               "sampled_sm_mhz": clocks.get("sm_mhz"), "clock_reasons": clocks.get("reasons")}
        out.update(gpu_info(dev.index))
        if wl in fd_set:
            out["directional_fd"] = directional_fd(mol, lay, dm_dev)
        print(json.dumps(out), flush=True)
        lay._cache.clear()
        del eng
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
