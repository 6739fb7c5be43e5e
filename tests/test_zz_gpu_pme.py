"""PME on the device (SURVEY.md §8(f)-3) against OpenMM's goldens for 6mrr and the reference's 3-water case, at the
reference's own tolerances (test/protein.jl:263-275, :277-299; test/interactions.jl:1683-1697).

The checker these mirror, oracle/pme.py, is pinned on the CPU (tests/test_oracle.py::test_6mrr_all_pme_openmm_golden,
::test_6mrr_vv_100steps_openmm_trajectory)."""
import os

import numpy as np
import pytest

import mbhelpers as H
import mollyb200 as mb

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_6mrr_all_pme_exact_openmm_golden_f64(golden_6mrr):
    """LJ + CoulombEwald(exact erfc) + bonded + PME + EwaldExclusion + LJDispersionCorrection, f64:
    max |dF| < 1e-7 kJ/mol/nm, |dE| < 1e-5 kJ/mol (test/protein.jl:267, :274)."""
    g = golden_6mrr
    s = H.sixmrr_pme_system(g, np.float64, exact=True)
    f, e = mb.forces_energy(s)
    err = np.linalg.norm(f[g["openmm_sample"]] - g["forces_all_pme_exact"], axis=1).max()
    de = e - float(g["energy_all_pme_exact"])
    print(f"[6mrr all_pme_exact f64] max|dF| = {err:.3e} kJ/mol/nm (bar 1e-7)  dE = {de:.3e} kJ/mol (bar 1e-5)")
    assert err < 1e-7 and abs(de) < 1e-5
    assert np.abs(mb.forces(s) - f).max() < 1e-9  # forces(sys) = the same sum of pairwise + specific + general
    s.close()


def test_6mrr_all_pme_approx_erfc_openmm_golden_f64(golden_6mrr):
    """The reference's default CoulombEwald (approximate_erfc=true): 1e-3 kJ/mol/nm, 0.2 kJ/mol (test/protein.jl:267, :274)."""
    g = golden_6mrr
    s = H.sixmrr_pme_system(g, np.float64, exact=False)
    f, e = mb.forces_energy(s)
    err = np.linalg.norm(f[g["openmm_sample"]] - g["forces_all_pme"], axis=1).max()
    de = e - float(g["energy_all_pme"])
    print(f"[6mrr all_pme (approximate erfc) f64] max|dF| = {err:.3e} (bar 1e-3)  dE = {de:.3e} (bar 0.2)")
    assert err < 1e-3 and abs(de) < 0.2
    assert err > 1e-6  # it IS the polynomial (oracle: 4.6e-4), not the exact function
    s.close()


def test_6mrr_pme_vv_100steps_openmm_trajectory_f64(golden_6mrr):
    """simulate!(sys_pme_exact, VelocityVerlet(dt=0.0005), 100) from velocities_300K vs OpenMM's coordinates_100steps /
    velocities_100steps: max |dx| < 1e-10 nm, max |dv| < 1e-7 nm/ps (test/protein.jl:277-299)."""
    g = golden_6mrr
    s = H.sixmrr_pme_system(g, np.float64, exact=True, velocities=g["velocities_300K"])
    assert abs(mb.kinetic_energy(s) - 65521.87288132431) < 1.5e-8 * 65521.87288132431
    e_tot = mb.potential_energy(s) + mb.kinetic_energy(s)
    assert abs(e_tot - 96522.24858589929) < 1.5e-8 * 96522.24858589929  # total_energy(sys_pme_exact), test/protein.jl:285
    mb.simulate(s, mb.VelocityVerlet(dt=0.0005), 100)
    box = g["box"]
    x_ref = g["coordinates_100steps"] - np.floor(g["coordinates_100steps"] / box) * box
    d = s.coords[g["openmm_sample"]] - x_ref
    d -= box * np.round(d / box)
    dx = np.linalg.norm(d, axis=1).max()
    dv = np.linalg.norm(s.velocities[g["openmm_sample"]] - g["velocities_100steps"], axis=1).max()
    st = s.stats()
    print(f"[6mrr PME VV 100 steps f64 vs OpenMM] dx = {dx:.3e} nm (bar 1e-10)  dv = {dv:.3e} nm/ps (bar 1e-7) "
          f"rebuilds={st['n_rebuilds']} graph={st['graph_mode']}")
    assert dx < 1e-10 and dv < 1e-7
    s.close()


@pytest.mark.parametrize("dtype,tol_f,tol_e", [(np.float64, 1e-7, 1e-8), (np.float32, 5e-4, 2e-4)])
def test_water3_pme_openmm_literals(dtype, tol_f, tol_e):
    """The reference's small PME case (test/interactions.jl:1683-1697): 3 waters, orthorhombic box, all-pairs path.
    f32 bars are the reference's own (5e-4 kJ/mol/nm, 2e-4 kJ/mol); f64 is held to the oracle's 1e-7 / 1e-8."""
    w = dict(np.load(os.path.join(ROOT, "tests", "golden", "water3.npz")))
    atoms = mb.atoms_from_arrays(w["mass"], w["charge"], w["sigma"], w["eps"], dtype)
    s = mb.System(atoms=atoms, coords=w["coords"].astype(dtype), boundary=mb.CubicBoundary(*w["box"]),
                  pairwise_inters=(mb.CoulombEwald(dist_cutoff=0.9, error_tol=0.0005, use_neighbors=True, approximate_erfc=False),),
                  neighbor_finder=mb.GPUNeighborFinder(dist_cutoff=0.9, excluded_pairs=w["excluded"] + 1),
                  dtype=dtype, general_inters=(mb.PME(dist_cutoff=0.9, error_tol=0.0005, excluded_pairs=w["excluded"] + 1),))
    f, e = mb.forces_energy(s)
    err = np.linalg.norm(f - w["forces_pme"], axis=1).max()
    print(f"[water3 {np.dtype(dtype).name}] max|dF| = {err:.3e} dE = {e - float(w['energy_pme']):.3e}")
    assert err < tol_f and abs(e - float(w["energy_pme"])) < tol_e
    s.close()


def test_c5_pme_total_energy_f64(golden_6mrr):
    """BASELINE config 5 on the system the reference ships goldens for (SURVEY.md section 8d: 6mrr with :pme, Float64): total energy
    over 0.2 ps of VelocityVerlet at two step sizes. The reference's energy-conservation protocol (test/energy_conservation.jl) is
    the soft LJ system of tests/test_gpu_parity.py::test_energy_conservation_reference_protocol, which passes at its 5e-4 kJ/mol
    bar; for a solvated protein it states no bar. Measured here (B200): E - E0 = -984 kJ/mol (1.5 % of KE) at dt 0.5 fs and
    -527 kJ/mol at dt 0.25 fs: an O(dt^2) part (this start - flexible TIP3P with velocities_300K - is off the integrator's shadow
    Hamiltonian while the O-H stretches thermalise) plus a step-size-independent part of about -380 kJ/mol that the truncated
    (not shifted) LJ / Ewald real-space energies at 1.0 nm allow. The same run with the reaction-field cutoff instead of PME, with
    or without CM removal, in one call or in ten gives the same curve (scripts/diag_c5.py), and OpenMM's own 100-step state,
    reproduced to 1e-10 nm by the trajectory test above, carries the same +85 kJ/mol. Asserted: bounded, and smaller with the
    smaller step."""
    g = golden_6mrr

    def drift(dt, n_steps):
        s = H.sixmrr_pme_system(g, np.float64, exact=True, velocities=g["velocities_300K"])
        ke0 = mb.kinetic_energy(s)
        e0 = mb.potential_energy(s) + ke0
        mb.simulate(s, mb.VelocityVerlet(dt=dt), n_steps)
        de = mb.potential_energy(s) + mb.kinetic_energy(s) - e0
        s.close()
        return de, ke0

    (d1, ke0), (d2, _) = drift(0.0005, 400), drift(0.00025, 800)
    print(f"[C5: 6mrr PME f64 NVE, 0.2 ps] E - E0 = {d1:.3f} kJ/mol at dt 0.5 fs ({abs(d1) / ke0:.2e} of KE), {d2:.3f} kJ/mol at dt 0.25 fs, "
          f"ratio {d1 / d2:.2f}")
    assert abs(d1) < 0.03 * ke0 and abs(d2) < abs(d1) and 1.3 < d1 / d2 < 5.0
