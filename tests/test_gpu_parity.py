"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs,
against the reference's golden vectors (tests/golden), and size-independent properties at full size.

Tolerances (stated per quantity):
  f64: per-atom force |dF| <= 1e-9 * max|F| + 1e-9 ; energy rel 1e-11 — same arithmetic, different order
       (the reference's own CPU-vs-GPU bar is rtol 1e-8, test/gpu_consistency.jl:43-49)
  f32: per-atom force |dF| <= 5e-5 * max|F| + 2e-3 kJ/mol/nm ; energy rel 2e-6 vs the f64 oracle on the
       same f32-rounded inputs (the reference accepts 5e-4 kJ/mol on E and 1e-4 nm on coords for its f32
       GPU path, test/simulation.jl:1246-1252)
  OpenMM goldens (6mrr, f64): max |dF| < 1e-7 kJ/mol/nm, |dE| < 1e-5 kJ/mol (test/protein.jl:263-275)
"""
import numpy as np
import pytest

import mbhelpers as H
import mollyb200 as mb
from oracle import oracle as o

pytestmark = pytest.mark.gpu


def _tol(dtype, fmax):
    return (1e-9 * fmax + 1e-9) if np.dtype(dtype) == np.float64 else (5e-5 * fmax + 2e-3)


def _etol(dtype, e):
    return (1e-11 if np.dtype(dtype) == np.float64 else 2e-6) * max(abs(e), 1.0)


def _boundary_atoms(orc, x64, o_inters, delta=3e-6):
    """Atoms that own a pair sitting on a cutoff within f32 rounding of r^2, where a DistanceCutoff /
    reaction-field force is discontinuous (it jumps by F(rc) ~ 1-2 kJ/mol/nm for CRF with water charges), and
    a bound on that jump. The reference has the same sensitivity between its f32 and f64 paths."""
    n = len(x64)
    count = np.zeros(n)
    for rc in sorted({it.r_cut for it in o_inters if it.r_cut > 0}):
        hi = orc.neighbor_list(x64, rc * (1 + delta))
        lo = orc.neighbor_list(x64, rc * (1 - delta))
        key = lambda a: set(map(tuple, a[:, :2].tolist()))
        for i, j in key(hi) - key(lo):
            count[i] += 1
            count[j] += 1
    return count


def _cutoff_force_bound(sysd, o_inters):
    """max |F(rc)| of a single pair over the interaction tuple."""
    b = 0.0
    qmax = np.abs(sysd["charge"]).max()
    for it in o_inters:
        rc = it.r_cut
        if rc <= 0:
            continue
        if it.kind == o.LJ and it.cutoff_kind == o.CUT_DISTANCE:
            sig, eps = sysd["sigma"].max(), sysd["eps"].max()
            s6 = (sig / rc) ** 6
            b += abs(24 * eps / rc * (2 * s6 * s6 - s6))
        elif it.kind == o.CRF:
            e = it.solvent_dielectric
            krf = (1 / rc ** 3) * (e - 1) / (2 * e + 1)
            b += it.coulomb_const * qmax * qmax * abs(1 / rc ** 2 - 2 * krf * rc)
        elif it.kind in (o.COULOMB, o.EWALD_REAL) and it.cutoff_kind == o.CUT_DISTANCE:
            b += it.coulomb_const * qmax * qmax / rc ** 2
    return b


def _pairwise_forces(s):
    """pairwise_forces_loop_gpu! seam only (mb_forces), whatever else the System carries."""
    fs = np.zeros((s.n, 3), s.dtype)
    mb.capi.check(s._L.mb_forces(s.engine(), s.coords.ctypes.data, fs.ctypes.data, None, 0))
    return fs


def _check(sysd, mb_inters, o_inters, dtype, r_list=0.0, expect_path=None, label=""):
    xin = sysd["coords"].astype(dtype)
    sd = dict(sysd, coords=xin)
    s = H.make_system(sd, mb_inters, dtype, r_list=r_list)
    orc = H.make_oracle(sd, o_inters, dtype=np.float64)
    f_ref, e_ref, vir_ref = orc.forces_allpairs(xin.astype(np.float64), virial=True)
    f = mb.forces(s)
    e = mb.potential_energy(s)
    f2, vir = mb.forces_virial(s)
    st = s.stats()
    if expect_path is not None:
        assert st["path"] == expect_path, st
    fmax = np.abs(f_ref).max()
    err = np.abs(f.astype(np.float64) - f_ref).max()
    print(f"[{label}] n={sysd['n']} dtype={np.dtype(dtype).name} path={st['path']} bricks={st['n_bricks']} "
          f"brick={st['brick_dims']} stride={st['list_stride']} maxnb={st['max_neighbors']} halo={st['max_halo']} "
          f"max|dF|={err:.3e} (max|F|={fmax:.3e}) dE={e - e_ref:.3e} (E={e_ref:.6e})")
    vtol = (1e-9 if np.dtype(dtype) == np.float64 else 1e-4) * max(np.abs(vir_ref).max(), 1.0)
    verr = np.abs(vir.astype(np.float64) - vir_ref).max()
    ferr2 = np.abs(f2.astype(np.float64) - f.astype(np.float64)).max()
    print(f"    virial err={verr:.3e} (tol {vtol:.3e}) |f(force-only) - f(force+virial)|={ferr2:.3e} repeat-equal={np.array_equal(f, mb.forces(s))}")
    if np.dtype(dtype) == np.float32 and err > _tol(dtype, fmax):
        # pairs sitting on the cutoff within f32 rounding may land on either side: allow one F(rc) jump each
        nb_pairs = _boundary_atoms(orc, xin.astype(np.float64), o_inters)
        fc = _cutoff_force_bound(sysd, o_inters)
        per_atom = np.abs(f.astype(np.float64) - f_ref).max(axis=1)
        allowed = _tol(dtype, fmax) + nb_pairs * fc
        print(f"    cutoff-boundary atoms: {int((nb_pairs > 0).sum())}; atoms over the plain tolerance: "
              f"{int((per_atom > _tol(dtype, fmax)).sum())}; F(rc) bound {fc:.3f}; "
              f"max err off-boundary={per_atom[nb_pairs == 0].max():.3e}")
        assert (per_atom <= allowed).all()
    else:
        assert err <= _tol(dtype, fmax)
    assert abs(e - e_ref) <= _etol(dtype, e_ref)
    assert np.array_equal(f, mb.forces(s))  # deterministic: same kernel, no atomics
    assert ferr2 <= _tol(dtype, fmax)       # the energy/virial variant may contract FMAs differently
    assert verr <= vtol
    s.close()
    return f, e


# ---------------------------------------------------------------------------------------------------
# all-pairs path (config 1 semantics)
# ---------------------------------------------------------------------------------------------------
def test_pair_known_answers_through_abi():
    # test/interactions.jl:61-82, :374-395 evaluated by the CUDA kernels
    def pair(inter, r, q=0.0):
        atoms = mb.atoms_from_arrays([10, 10], [q, q], [0.3, 0.3], [0.2, 0.2], np.float64)
        s = mb.System(atoms=atoms, coords=np.array([[1.0, 1, 1], [1.0 + r, 1, 1]]), boundary=mb.CubicBoundary(5.0),
                      pairwise_inters=(inter,), dtype=np.float64)
        f, e = mb.forces(s)[1, 0], mb.potential_energy(s)
        s.close()
        return f, e
    f, e = pair(mb.LennardJones(), 0.3)
    assert abs(f - 16.0) < 1e-9 and abs(e) < 1e-9
    f, e = pair(mb.LennardJones(), 0.4)
    assert abs(f + 1.375509739) < 1e-9 and abs(e + 0.1170417309) < 1e-9
    f, e = pair(mb.Coulomb(), 0.3, 1.0)
    assert abs(f - 1543.727311) < 1e-5 and abs(e - 463.1181933) < 1e-5
    f, e = pair(mb.CoulombReactionField(dist_cutoff=1.0), 1.2, 1.0)
    assert f == 0.0 and e == 0.0


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_readme_system_allpairs(dtype):
    sd = H.readme_system(100, 2.0, seed=1)
    _check(sd, (mb.LennardJones(),), [o.Inter(o.LJ)], dtype, expect_path=0, label="C1 readme")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("cut", ["distance", "shifted_potential", "shifted_force"])
def test_molecular_allpairs_exceptions(dtype, cut):
    # box smaller than 2.5 r_list -> the all-pairs kernel serves neighbour-list interactions (exclusions apply)
    sd = H.molecular_system(150, [3.0, 3.2, 3.4], seed=11)
    mcut = {"distance": mb.DistanceCutoff, "shifted_potential": mb.ShiftedPotentialCutoff,
            "shifted_force": mb.ShiftedForceCutoff}[cut](1.2)
    ocut = {"distance": o.CUT_DISTANCE, "shifted_potential": o.CUT_SHIFTED_POTENTIAL,
            "shifted_force": o.CUT_SHIFTED_FORCE}[cut]
    _check(sd, (mb.LennardJones(cutoff=mcut, weight_special=0.5, use_neighbors=True),
                mb.Coulomb(cutoff=mcut, weight_special=0.8333, use_neighbors=True)),
           [o.Inter(o.LJ, ocut, 1.2, weight_special=0.5, use_neighbors=True),
            o.Inter(o.COULOMB, ocut, 1.2, weight_special=0.8333, use_neighbors=True)],
           dtype, r_list=1.3, expect_path=0, label=f"molecular all-pairs {cut}")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_mixed_nl_and_nonl_interactions(dtype):
    """use_neighbors=false interactions ignore the exclusion / special masks (src/force.jl:828-855):
    LJ through the list (with exclusions), Coulomb over all pairs (without)."""
    sd = H.molecular_system(150, [3.0, 3.2, 3.4], seed=13)
    sd = dict(sd, charge=sd["charge"] * 0.1)
    _check(sd, (mb.LennardJones(cutoff=mb.DistanceCutoff(1.2), weight_special=0.5, use_neighbors=True),
                mb.Coulomb(cutoff=mb.DistanceCutoff(1.2), weight_special=0.8333, use_neighbors=False)),
           [o.Inter(o.LJ, o.CUT_DISTANCE, 1.2, weight_special=0.5, use_neighbors=True),
            o.Inter(o.COULOMB, o.CUT_DISTANCE, 1.2, weight_special=0.8333, use_neighbors=False)],
           dtype, r_list=1.3, expect_path=0, label="mixed nl/non-nl")


# ---------------------------------------------------------------------------------------------------
# brick / neighbour-list path
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("cells", [6, 9])
def test_lj_fluid_brick_path(dtype, cells):
    sd = H.lj_fluid(cells, seed=42, dtype=np.float64)  # 864 / 2916 atoms at the C2 density, rc 1.2 nm
    rc = 1.2 if cells >= 9 else 0.9
    _check(sd, (mb.LennardJones(cutoff=mb.DistanceCutoff(rc), use_neighbors=True),),
           [o.Inter(o.LJ, o.CUT_DISTANCE, rc, use_neighbors=True)], dtype, r_list=rc + 0.1, expect_path=1,
           label=f"LJ fluid {cells}")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_lj_fluid_16k(dtype):
    sd = H.lj_fluid(16, seed=42, dtype=np.float64)  # 16384 atoms, box 9.19 nm
    _check(sd, (mb.LennardJones(cutoff=mb.DistanceCutoff(1.2), use_neighbors=True),),
           [o.Inter(o.LJ, o.CUT_DISTANCE, 1.2, use_neighbors=True)], dtype, r_list=1.3, expect_path=1, label="LJ 16k")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("coul", ["crf", "coulomb_sf", "ewald", "ewald_approx"])
def test_molecular_brick_path(dtype, coul):
    sd = H.molecular_system(1000, [5.1, 5.4, 5.8], seed=5)  # 4000 atoms, orthorhombic, mixed types, charges
    lj_m = mb.LennardJones(cutoff=mb.DistanceCutoff(1.0), use_neighbors=True, weight_special=0.5)
    lj_o = o.Inter(o.LJ, o.CUT_DISTANCE, 1.0, weight_special=0.5, use_neighbors=True)
    if coul == "crf":
        c_m = mb.CoulombReactionField(dist_cutoff=1.0, use_neighbors=True, weight_special=0.8333)
        c_o = o.Inter(o.CRF, o.CUT_DISTANCE, 1.0, weight_special=0.8333, use_neighbors=True)
    elif coul == "coulomb_sf":
        c_m = mb.Coulomb(cutoff=mb.ShiftedForceCutoff(1.0), use_neighbors=True, weight_special=0.8333)
        c_o = o.Inter(o.COULOMB, o.CUT_SHIFTED_FORCE, 1.0, weight_special=0.8333, use_neighbors=True)
    else:
        approx = coul == "ewald_approx"  # approximate_erfc=true is the reference's default (coulomb.jl:1331)
        c_m = mb.CoulombEwald(dist_cutoff=1.0, use_neighbors=True, weight_special=0.8333, approximate_erfc=approx)
        alpha = float(np.sqrt(-np.log(2 * 5e-4)) / 1.0)
        c_o = o.Inter(o.EWALD_REAL, o.CUT_DISTANCE, 1.0, weight_special=0.8333, ewald_alpha=alpha, use_neighbors=True,
                      approx_erfc=approx)
    _check(sd, (lj_m, c_m), [lj_o, c_o], dtype, r_list=1.1, expect_path=1, label=f"molecular brick {coul}")


@pytest.mark.parametrize("name", ["lj_only", "coul_only"])
def test_6mrr_openmm_golden_f64(golden_6mrr, name):
    """The reference's own GPU bar (test/protein.jl:356-360): CUDA f64 vs OpenMM Reference platform."""
    g = golden_6mrr
    box = g["box"]
    x = g["coords"] - np.floor(g["coords"] / box) * box
    if name == "lj_only":
        inter = mb.LennardJones(cutoff=mb.DistanceCutoff(1.0), use_neighbors=True, weight_special=float(g["lj14scale"]))
    else:
        inter = mb.CoulombReactionField(dist_cutoff=1.0, use_neighbors=True, weight_special=float(g["coulomb14scale"]))
    atoms = mb.atoms_from_arrays(g["mass"], g["charge"], g["sigma"], g["eps"], np.float64)
    nf = mb.GPUNeighborFinder(dist_cutoff=1.2, excluded_pairs=g["excluded"] + 1, special_pairs=g["special"] + 1)
    # lj_only carries sys.general_inters = (LJDispersionCorrection,) in the reference's test (test/protein.jl:247-248)
    gis = (mb.LJDispersionCorrection(1.0),) if name == "lj_only" else ()
    s = mb.System(atoms=atoms, coords=x, boundary=mb.CubicBoundary(*box), pairwise_inters=(inter,), neighbor_finder=nf,
                  dtype=np.float64, general_inters=gis)
    f = mb.forces(s)
    e = mb.potential_energy(s)
    st = s.stats()
    if name == "lj_only":  # the product's correction equals the oracle's restatement of the constructor
        e_pair = np.zeros(1)
        mb.capi.check(s._L.mb_energy(s.engine(), s.coords.ctypes.data, e_pair.ctypes.data, 0))
        assert abs((e - e_pair[0]) - o.lj_dispersion_correction_energy(g["sigma"], g["eps"], box, 1.0)) < 1e-9
    err = np.linalg.norm(f[g["openmm_sample"]] - g[f"forces_{name}"], axis=1).max()
    print(f"[6mrr {name}] path={st['path']} brick={st['brick_dims']} maxnb={st['max_neighbors']} "
          f"pairs={st['n_pairs_in_list']} max|dF|={err:.3e} dE={e - float(g[f'energy_{name}']):.3e}")
    assert st["path"] == 1
    assert err < 1e-7
    assert abs(e - float(g[f"energy_{name}"])) < 1e-5
    if name == "lj_only":
        # full-shell list at 1.2 nm holds every eligible pair twice: 2 x 4 602 420 (test/basic.jl:592)
        assert st["n_pairs_in_list"] == 2 * 4602420
    s.close()


def test_6mrr_f32_vs_oracle(golden_6mrr):
    g = golden_6mrr
    box = g["box"]
    x = (g["coords"] - np.floor(g["coords"] / box) * box).astype(np.float32)
    sd = dict(n=len(x), box=box, coords=x, velocities=g["velocities_300K"], mass=g["mass"], charge=g["charge"],
              sigma=g["sigma"], eps=g["eps"], excluded=g["excluded"], special=g["special"])
    _check(sd, (mb.LennardJones(cutoff=mb.DistanceCutoff(1.0), use_neighbors=True, weight_special=0.5),
                mb.CoulombReactionField(dist_cutoff=1.0, use_neighbors=True, weight_special=float(g["coulomb14scale"]))),
           [o.Inter(o.LJ, o.CUT_DISTANCE, 1.0, weight_special=0.5, use_neighbors=True),
            o.Inter(o.CRF, o.CUT_DISTANCE, 1.0, weight_special=float(g["coulomb14scale"]), use_neighbors=True)],
           np.float32, r_list=1.15, expect_path=1, label="6mrr LJ+CRF f32")


def test_forces_track_moving_coordinates_and_rebuild():
    """Buffer reuse across calls (test/gpu_consistency.jl:451-492): move atoms a little (no rebuild), then a lot
    (forces a rebuild), including periodic wrapping by the caller."""
    sd = H.lj_fluid(9, seed=5, dtype=np.float64)
    inter_m = (mb.LennardJones(cutoff=mb.DistanceCutoff(1.0), use_neighbors=True),)
    inter_o = [o.Inter(o.LJ, o.CUT_DISTANCE, 1.0, use_neighbors=True)]
    s = H.make_system(sd, inter_m, np.float64, r_list=1.2)
    orc = H.make_oracle(sd, inter_o)
    rng = np.random.default_rng(0)
    x = sd["coords"].copy()
    rebuilds = []
    for it, amp in enumerate([0.0, 0.01, 0.01, 0.3, 0.01]):
        x = x + rng.normal(0, amp, x.shape) if amp else x
        x = x - np.floor(x / sd["box"]) * sd["box"]  # caller wraps, atoms jump across the box
        s.coords = x.copy()
        f = mb.forces(s)
        f_ref, _, _ = orc.forces_allpairs(x)
        assert np.abs(f - f_ref).max() <= 1e-9 * np.abs(f_ref).max() + 1e-9, it
        rebuilds.append(s.stats()["n_rebuilds"])
    print("rebuild counts:", rebuilds)
    assert rebuilds[1] == rebuilds[0] and rebuilds[3] > rebuilds[2]
    s.close()


# ---------------------------------------------------------------------------------------------------
# bonded terms + the whole 6mrr :cutoff system (SURVEY.md §8f-1)
# ---------------------------------------------------------------------------------------------------
def test_6mrr_all_cut_openmm_golden_f64(golden_6mrr):
    """LJ + CRF + HarmonicBond + HarmonicAngle + PeriodicTorsion (propers + impropers) on the GPU vs OpenMM's
    forces_all_cut / energy_all_cut (test/protein.jl:263-275: 1e-7 kJ/mol/nm, 1e-5 kJ/mol)."""
    g = golden_6mrr
    s = H.sixmrr_system(g, np.float64, r_list=1.2, dispersion=True)
    f, e = mb.forces_energy(s)
    err = np.linalg.norm(f[g["openmm_sample"]] - g["forces_all_cut"], axis=1).max()
    print(f"[6mrr all_cut f64] max|dF|={err:.3e} dE={e - float(g['energy_all_cut']):.3e}")
    assert err < 1e-7
    assert abs(e - float(g["energy_all_cut"])) < 1e-5
    # forces(sys) / potential_energy(sys) route through the same all-interaction entry point
    assert np.abs(mb.forces(s) - f).max() < 1e-9 and abs(mb.potential_energy(s) - e) < 1e-9 * abs(e)
    # bonded-only parity: pairwise-only seam (mb_forces) subtracted
    f_pair = _pairwise_forces(s)
    fb_ref = sum(g[f"forces_{k}_only"] for k in ("bond", "angle", "proptor", "improptor"))
    assert np.linalg.norm((f - f_pair)[g["openmm_sample"]] - fb_ref, axis=1).max() < 1e-7
    s.close()


def test_6mrr_all_cut_f32_vs_oracle(golden_6mrr):
    g = golden_6mrr
    s = H.sixmrr_system(g, np.float32, r_list=1.15)
    orc, sd = H.sixmrr_oracle(g)
    x32 = sd["coords"].astype(np.float32)
    f_ref, _, _ = orc.forces_allpairs(x32.astype(np.float64), energy=False)
    fb, eb = H.bonded_forces_oracle(g, x32.astype(np.float64))
    f, e = mb.forces_energy(s)
    fb_gpu = f - _pairwise_forces(s)
    berr = np.abs(fb_gpu - fb).max()
    print(f"[6mrr bonded f32] max|dF_bonded|={berr:.3e} (max|F_bonded|={np.abs(fb).max():.3e})")
    assert berr < 1e-4 * np.abs(fb).max() + 5e-2  # stiff bonds (k ~ 4.6e5): (r - r0) cancellation in f32
    s.close()


def test_6mrr_vv_with_bonded_f64_matches_oracle(golden_6mrr):
    """The benchmark/protein.jl system (dt 0.5 fs, no coupling) for 20 steps vs the oracle's VV loop."""
    g = golden_6mrr
    s = H.sixmrr_system(g, np.float64, r_list=1.2, n_steps=10)
    sd = H.sixmrr_description(g)
    x_ref, v_ref = H.oracle_vv_with_bonded(g, sd["coords"], sd["velocities"], 0.0005, 20, r_list=1.2, nl_every=10)
    mb.simulate(s, mb.VelocityVerlet(dt=0.0005), 20)
    ex, ev = _pos_err(s.coords, x_ref, sd["box"]), np.abs(s.velocities - v_ref).max()
    print(f"[6mrr VV bonded f64] dx={ex:.3e} dv={ev:.3e} graph={s.stats()['graph_mode']}")
    assert ex < 1e-9 and ev < 1e-6
    s.close()


def test_6mrr_dynamics_f32_tracks_f64(golden_6mrr):
    """benchmark/protein.jl's run (flexible water, dt 0.5 fs, NVE): the equilibrated-with-constraints start structure
    carries 1.6e5 kJ/mol of bond energy, so the system heats (329 K -> ~580 K in 500 steps) while total energy is
    conserved. Check conservation in f64 and that f32 follows f64."""
    g = golden_6mrr
    res = {}
    for dtype in (np.float64, np.float32):
        s = H.sixmrr_system(g, dtype, r_list=1.12)
        _, pe0 = mb.forces_energy(s)
        e0 = pe0 + mb.kinetic_energy(s)
        mb.simulate(s, mb.VelocityVerlet(dt=0.0005), 300)
        _, pe1 = mb.forces_energy(s)
        ke1 = mb.kinetic_energy(s)
        res[dtype] = (e0, pe1 + ke1, mb.temperature(s), s.stats()["n_rebuilds"])
        assert np.isfinite(s.coords).all()
        s.close()
    print(f"[6mrr NVE 300 steps] f64 E0={res[np.float64][0]:.1f} E1={res[np.float64][1]:.1f} T={res[np.float64][2]:.1f}; "
          f"f32 E1={res[np.float32][1]:.1f} T={res[np.float32][2]:.1f} rebuilds={res[np.float64][3]}")
    e0, e1, t64, _ = res[np.float64]
    assert abs(e1 - e0) < 0.01 * abs(e0)        # VV at 0.5 fs with 3000 cm^-1 O-H stretches: ~0.6 % over 300 steps
    assert abs(res[np.float32][2] - t64) < 2.0    # K
    assert abs(res[np.float32][1] - e1) < 5e-4 * abs(e1)


def test_6mrr_andersen_runs(golden_6mrr):
    """Config 3 (VelocityVerlet + AndersenThermostat(300 K, 1 ps), f32) runs and stays finite; resampled atoms follow
    the target distribution only on the ps time scale, so no temperature bar here (see test_andersen_thermostat_statistics)."""
    g = golden_6mrr
    s = H.sixmrr_system(g, np.float32, r_list=1.12)
    mb.simulate(s, mb.VelocityVerlet(dt=0.0005, coupling=mb.AndersenThermostat(300.0, 1.0)), 200, rng=np.random.default_rng(3))
    assert np.isfinite(s.coords).all() and np.isfinite(s.velocities).all()
    assert 250.0 < mb.temperature(s) < 700.0
    s.close()


# ---------------------------------------------------------------------------------------------------
# VelocityVerlet
# ---------------------------------------------------------------------------------------------------
def _pos_err(a, b, box):
    d = a.astype(np.float64) - b.astype(np.float64)
    d -= box * np.round(d / box)
    return np.abs(d).max()


@pytest.mark.parametrize("policy", [0, 10])
def test_vv_lj_fluid_f64_matches_oracle(policy):
    sd = H.lj_fluid(9, seed=7, dtype=np.float64, temp=120.0)
    rc, rl, dt, n = 1.0, 1.1, 0.002, 60  # skin 0.1 nm: the displacement trigger fires inside the run
    s = H.make_system(sd, (mb.LennardJones(cutoff=mb.DistanceCutoff(rc), use_neighbors=True),), np.float64, r_list=rl,
                      n_steps=policy)
    orc = H.make_oracle(sd, [o.Inter(o.LJ, o.CUT_DISTANCE, rc, use_neighbors=True)])
    x_ref, v_ref, _ = orc.simulate_vv(sd["coords"], sd["velocities"], dt, n, remove_cm_every=1, r_list=rl, nl_every=10)
    mb.simulate(s, mb.VelocityVerlet(dt=dt), n)
    st = s.stats()
    ex, ev = _pos_err(s.coords, x_ref, sd["box"]), np.abs(s.velocities - v_ref).max()
    print(f"[VV LJ f64 policy={policy}] rebuilds={st['n_rebuilds']} violations={st['violations']} dx={ex:.3e} dv={ev:.3e}")
    # a DistanceCutoff force is discontinuous at rc, so pairs crossing the cutoff amplify rounding; bars follow
    # test/simulation.jl:1246-1252 (1e-4 nm) tightened for f64
    assert ex < 1e-7 and ev < 1e-5
    assert (s.coords >= 0).all() and (s.coords < sd["box"]).all()
    assert np.abs((sd["mass"][:, None] * s.velocities).sum(0)).max() < 1e-8
    if policy == 0:
        assert st["n_rebuilds"] >= 2 and st["violations"] == 0
    s.close()


def test_vv_molecular_f64_matches_oracle():
    sd = H.molecular_system(729, [5.1, 5.4, 5.8], seed=5, stable=True)
    lj_m = mb.LennardJones(cutoff=mb.ShiftedForceCutoff(1.0), use_neighbors=True, weight_special=0.5)
    c_m = mb.CoulombReactionField(dist_cutoff=1.0, use_neighbors=True, weight_special=0.8333)
    lj_o = o.Inter(o.LJ, o.CUT_SHIFTED_FORCE, 1.0, weight_special=0.5, use_neighbors=True)
    c_o = o.Inter(o.CRF, o.CUT_DISTANCE, 1.0, weight_special=0.8333, use_neighbors=True)
    s = H.make_system(sd, (lj_m, c_m), np.float64, r_list=1.15)
    orc = H.make_oracle(sd, [lj_o, c_o])
    dt, n = 0.0005, 40
    x_ref, v_ref, _ = orc.simulate_vv(sd["coords"], sd["velocities"], dt, n, remove_cm_every=1, r_list=1.15, nl_every=5)
    mb.simulate(s, mb.VelocityVerlet(dt=dt), n)
    ex, ev = _pos_err(s.coords, x_ref, sd["box"]), np.abs(s.velocities - v_ref).max()
    print(f"[VV molecular f64] dx={ex:.3e} dv={ev:.3e} rebuilds={s.stats()['n_rebuilds']}")
    assert ex < 1e-7 and ev < 1e-4
    s.close()


def test_vv_readme_allpairs_f64():
    sd = H.readme_system(100, 2.0, seed=1)
    s = H.make_system(sd, (mb.LennardJones(),), np.float64)
    orc = H.make_oracle(sd, [o.Inter(o.LJ)])
    x_ref, v_ref, _ = orc.simulate_vv(sd["coords"], sd["velocities"], 0.002, 100, remove_cm_every=1, r_list=0.0)
    mb.simulate(s, mb.VelocityVerlet(dt=0.002), 100)
    ex, ev = _pos_err(s.coords, x_ref, sd["box"]), np.abs(s.velocities - v_ref).max()
    print(f"[VV readme f64] dx={ex:.3e} dv={ev:.3e}")
    assert ex < 1e-9 and ev < 1e-8
    s.close()


def test_vv_f32_tracks_f64_oracle():
    sd = H.lj_fluid(9, seed=7, dtype=np.float64, temp=90.0)
    rc, rl, dt, n = 1.0, 1.2, 0.002, 50
    s = H.make_system(sd, (mb.LennardJones(cutoff=mb.ShiftedForceCutoff(rc), use_neighbors=True),), np.float32, r_list=rl)
    orc = H.make_oracle(dict(sd, coords=sd["coords"].astype(np.float32), velocities=sd["velocities"].astype(np.float32)),
                        [o.Inter(o.LJ, o.CUT_SHIFTED_FORCE, rc, use_neighbors=True)])
    x_ref, v_ref, _ = orc.simulate_vv(sd["coords"].astype(np.float32), sd["velocities"].astype(np.float32), dt, n,
                                      remove_cm_every=1, r_list=rl, nl_every=10)
    mb.simulate(s, mb.VelocityVerlet(dt=dt), n)
    ex = _pos_err(s.coords, x_ref, sd["box"])
    print(f"[VV LJ f32] dx={ex:.3e}")
    assert ex < 1e-4  # test/simulation.jl:1251
    s.close()


def test_vv_chunked_equals_single_call():
    """simulate!(n1) then simulate!(n2; init_step=n1) == simulate!(n1+n2) (state fully round-trips through the ABI)."""
    sd = H.lj_fluid(6, seed=3, dtype=np.float64)
    mk = lambda: H.make_system(sd, (mb.LennardJones(cutoff=mb.ShiftedForceCutoff(0.9), use_neighbors=True),),
                               np.float64, r_list=1.0)
    a, b = mk(), mk()
    mb.simulate(a, mb.VelocityVerlet(dt=0.002), 40)
    mb.simulate(b, mb.VelocityVerlet(dt=0.002), 25)
    mb.simulate(b, mb.VelocityVerlet(dt=0.002), 15, init_step=25)
    assert _pos_err(a.coords, b.coords, sd["box"]) < 1e-9
    assert np.abs(a.velocities - b.velocities).max() < 1e-8
    a.close(); b.close()


def test_andersen_thermostat_statistics():
    # test/coupling.jl:67-98: 9.5 K < <T> < 10.5 K, std < 1 K (here 2916 atoms, shorter run)
    sd = H.lj_fluid(9, seed=11, dtype=np.float64, temp=10.0)
    s = H.make_system(sd, (mb.LennardJones(cutoff=mb.ShiftedForceCutoff(1.0), use_neighbors=True),), np.float32, r_list=1.2)
    sim = mb.VelocityVerlet(dt=0.002, coupling=mb.AndersenThermostat(10.0, 0.1))
    temps = []
    rng = np.random.default_rng(1)
    mb.simulate(s, sim, 300, rng=rng)
    for k in range(20):
        mb.simulate(s, sim, 25, init_step=300 + 25 * k, rng=rng)
        temps.append(mb.temperature(s))
    print(f"[Andersen] <T>={np.mean(temps):.3f} std={np.std(temps):.3f}")
    assert 9.5 < np.mean(temps) < 10.5 and np.std(temps) < 1.0
    s.close()


def test_kinetic_energy_and_cm(golden_6mrr):
    g = golden_6mrr
    atoms = mb.atoms_from_arrays(g["mass"], g["charge"], g["sigma"], g["eps"], np.float64)
    s = mb.System(atoms=atoms, coords=g["coords"], boundary=mb.CubicBoundary(*g["box"]), velocities=g["velocities_300K"],
                  pairwise_inters=(mb.LennardJones(cutoff=mb.DistanceCutoff(1.0), use_neighbors=True),),
                  neighbor_finder=mb.GPUNeighborFinder(dist_cutoff=1.2), dtype=np.float64)
    assert abs(mb.kinetic_energy(s) - 65521.87288132431) < 1.5e-8 * 65521.87288132431  # test/protein.jl:284
    assert abs(mb.temperature(s) - 329.3202932884933) < 1.5e-8 * 329.3202932884933
    mb.remove_CM_motion(s)
    assert np.abs((g["mass"][:, None] * s.velocities).sum(0)).max() < 1e-8
    s.close()


# ---------------------------------------------------------------------------------------------------
# full-size properties (BASELINE config 2: 256 000 atoms, f32, rc 1.2 nm)
# ---------------------------------------------------------------------------------------------------
def test_c2_full_size_properties():
    sd = H.lj_fluid(40, seed=42, dtype=np.float32)
    assert sd["n"] == 256000
    inter = (mb.LennardJones(cutoff=mb.DistanceCutoff(1.2), use_neighbors=True),)
    s = H.make_system(sd, inter, np.float32, r_list=1.3)
    f = mb.forces(s)
    e = mb.potential_energy(s)
    st = s.stats()
    print(f"[C2] bricks={st['n_bricks']} brick={st['brick_dims']} stride={st['list_stride']} maxnb={st['max_neighbors']} "
          f"halo={st['max_halo']} pairs/atom={st['n_pairs_in_list'] / sd['n']:.1f} E={e:.6e}")
    # Newton's third law: forces sum to zero up to f32 rounding
    assert np.abs(f.astype(np.float64).sum(0)).max() < 1e-4 * np.abs(f).max() * np.sqrt(sd["n"])
    # determinism
    assert np.array_equal(f, mb.forces(s))
    # sampled parity: oracle forces on 64 atoms via a 20 000-atom neighbourhood is expensive; use translation
    # invariance instead: shifting every atom by the same vector (mod box) leaves forces unchanged up to rounding
    shift = np.array([3.3, -7.1, 11.9], np.float32)
    x2 = sd["coords"] + shift
    x2 = (x2 - np.floor(x2 / sd["box"]) * sd["box"]).astype(np.float32)
    s2 = H.make_system(dict(sd, coords=x2), inter, np.float32, r_list=1.3)
    f2 = mb.forces(s2)
    assert np.abs(f2 - f).max() < 2e-3 * np.abs(f).max()
    # permutation invariance: relabelling atoms permutes the forces
    perm = np.random.default_rng(0).permutation(sd["n"])
    s3 = H.make_system(dict(sd, coords=sd["coords"][perm]), inter, np.float32, r_list=1.3)
    f3 = mb.forces(s3)
    assert np.abs(f3 - f[perm]).max() < 1e-4 * np.abs(f).max()
    # pair count: in-cutoff neighbours per atom for rho = 21.105 nm^-3, r_list 1.3 -> 4/3 pi r^3 rho = 194.2
    assert abs(st["n_pairs_in_list"] / sd["n"] - 194.2) < 3.0
    for q in (s, s2, s3):
        q.close()


def test_c2_energy_conservation_f32():
    """NVE drift over 200 steps at full size with a shifted-force cutoff (continuous force)."""
    sd = H.lj_fluid(40, seed=42, dtype=np.float32)
    s = H.make_system(sd, (mb.LennardJones(cutoff=mb.ShiftedForceCutoff(1.2), use_neighbors=True),), np.float32, r_list=1.3)
    e0 = mb.potential_energy(s) + mb.kinetic_energy(s)
    mb.simulate(s, mb.VelocityVerlet(dt=0.002), 200)
    e1 = mb.potential_energy(s) + mb.kinetic_energy(s)
    ke = mb.kinetic_energy(s)
    st = s.stats()
    print(f"[C2 NVE] E0={e0:.4f} E1={e1:.4f} drift={(e1 - e0) / sd['n']:.3e} kJ/mol/atom KE={ke:.2f} rebuilds={st['n_rebuilds']}")
    assert abs(e1 - e0) / sd["n"] < 2e-3  # ~0.3 % of kT per atom at 90 K
    s.close()


# ---------------------------------------------------------------------------------------------------
# full-size parity against the oracle's neighbour-list path (the configs that carry the bench numbers)
# ---------------------------------------------------------------------------------------------------
def _full_size_vs_oracle(cells, label):
    """Forces + energy of the packed-f32 fast path at full size vs the f64 oracle on the same f32-rounded coordinates.
    Bar: the repo's f32 tolerance (5e-5 max|F| + 2e-3 kJ/mol/nm per component; pairs within f32 rounding of the cutoff
    may land on either side and are allowed one F(rc) jump each), energy rel 2e-6."""
    sd = H.lj_fluid(cells, seed=42, dtype=np.float32)
    inter = (mb.LennardJones(cutoff=mb.DistanceCutoff(1.2), use_neighbors=True),)
    o_inters = [o.Inter(o.LJ, o.CUT_DISTANCE, 1.2, use_neighbors=True)]
    s = H.make_system(sd, inter, np.float32, r_list=1.3)
    f = mb.forces(s)
    e = mb.potential_energy(s)
    st = s.stats()
    orc = H.make_oracle(sd, o_inters, dtype=np.float64)
    x64 = sd["coords"].astype(np.float64)
    nl = orc.neighbor_list(x64, 1.2 * (1 + 3e-6))
    f_ref, e_ref, _ = orc.forces_nl(x64, nl)
    fmax = np.abs(f_ref).max()
    per_atom = np.abs(f.astype(np.float64) - f_ref).max(axis=1)
    lo = orc.neighbor_list(x64, 1.2 * (1 - 3e-6))
    on_cut = np.zeros(sd["n"])
    key = lambda a: a[:, 0].astype(np.int64) * sd["n"] + a[:, 1]
    extra = nl[~np.isin(key(nl), key(lo))]
    np.add.at(on_cut, extra[:, 0], 1)
    np.add.at(on_cut, extra[:, 1], 1)
    fc = _cutoff_force_bound(sd, o_inters)
    print(f"[{label}] n={sd['n']} bricks={st['n_bricks']} brick={st['brick_dims']} in-cutoff pairs={len(lo)} "
          f"max|dF|={per_atom.max():.3e} (max|F|={fmax:.3e}) pairs on the cutoff={len(extra)} F(rc)={fc:.3e} "
          f"dE/E={(e - e_ref) / abs(e_ref):.3e}")
    assert (per_atom <= _tol(np.float32, fmax) + on_cut * fc).all()
    assert abs(e - e_ref) <= _etol(np.float32, e_ref)
    assert np.array_equal(f, mb.forces(s))
    return sd, s, orc


def test_c2_full_size_vs_oracle():
    """BASELINE config 2 (256 000 atoms, f32, rc 1.2 nm, brick 3x3x2): single evaluation, then 100 VelocityVerlet steps
    against the oracle's VV loop (bar: test/simulation.jl:1246-1252, 1e-4 nm for the f32 GPU path)."""
    sd, s, orc = _full_size_vs_oracle(40, "C2 full size")
    x_ref, v_ref, _ = orc.simulate_vv(sd["coords"], sd["velocities"], 0.002, 100, remove_cm_every=1, r_list=1.4, nl_every=10)
    mb.simulate(s, mb.VelocityVerlet(dt=0.002), 100)
    ex, ev = _pos_err(s.coords, x_ref, sd["box"]), np.abs(s.velocities - v_ref).max()
    st = s.stats()
    print(f"[C2 VV 100 steps f32 vs f64 oracle] dx={ex:.3e} nm dv={ev:.3e} nm/ps rebuilds={st['n_rebuilds']} graph={st['graph_mode']}")
    assert ex < 1e-4
    s.close()


def test_c4_full_size_vs_oracle():
    """BASELINE config 4 (1 000 188 atoms): single force + energy evaluation vs the oracle."""
    sd, s, _ = _full_size_vs_oracle(63, "C4 full size")
    assert sd["n"] == 1000188
    s.close()


# ---------------------------------------------------------------------------------------------------
# boundary contract details (SURVEY.md §8 A1, A2)
# ---------------------------------------------------------------------------------------------------
def test_forces_add_into_nonzero_fs_mat_and_device_pointers():
    """pairwise_forces_loop_gpu! ADDs into fs_mat (force.jl:1216 zeroes it first; the kernel contract is +=), for host
    and for device output arrays; mb_set_atoms accepts a device pointer (what the Julia shim passes: CuArray{Atom})."""
    import ctypes as C
    import torch
    sd = H.lj_fluid(9, seed=42, dtype=np.float64)
    inter = (mb.LennardJones(cutoff=mb.DistanceCutoff(1.0), use_neighbors=True),)
    s = H.make_system(sd, inter, np.float64, r_list=1.2)
    f0 = mb.forces(s)
    pre = np.random.default_rng(0).normal(size=f0.shape)
    fs = pre.copy()
    mb.capi.check(s._L.mb_forces(s.engine(), s.coords.ctypes.data, fs.ctypes.data, None, 0))
    assert np.abs(fs - (pre + f0)).max() <= 1e-12 * np.abs(f0).max()
    # device output + device coords
    xd = torch.from_numpy(s.coords).cuda()
    fd = torch.from_numpy(pre).cuda()
    mb.capi.check(s._L.mb_forces(s.engine(), xd.data_ptr(), fd.data_ptr(), None, 0))
    torch.cuda.synchronize()
    assert np.abs(fd.cpu().numpy() - (pre + f0)).max() <= 1e-12 * np.abs(f0).max()
    # energy ADD
    pe = np.array([7.5])
    mb.capi.check(s._L.mb_energy(s.engine(), s.coords.ctypes.data, pe.ctypes.data, 0))
    assert abs(pe[0] - 7.5 - mb.potential_energy(s)) < 1e-9 * abs(pe[0])
    # atoms from a device pointer: a second context fed the same AoS bytes from device memory
    L = s._L
    ctx = C.c_void_p()
    mb.capi.check(L.mb_ctx_create(0, 64, None, C.byref(ctx)))
    atoms_dev = torch.from_numpy(s.atoms.view(np.uint8).copy()).cuda()
    mb.capi.check(L.mb_set_atoms(ctx, s.n, atoms_dev.data_ptr()))
    mb.capi.check(L.mb_set_box(ctx, (C.c_double * 3)(*sd["box"])))
    d = inter[0].descriptor()
    mb.capi.check(L.mb_set_inters(ctx, 1, (mb.capi.MBInter * 1)(d)))
    mb.capi.check(L.mb_set_neighbor_policy(ctx, 1.2, 0))
    f2 = np.zeros_like(f0)
    mb.capi.check(L.mb_forces(ctx, s.coords.ctypes.data, f2.ctypes.data, None, 0))
    assert np.array_equal(f2, f0)
    L.mb_ctx_destroy(ctx)
    s.close()


# ---------------------------------------------------------------------------------------------------
# two-point cutoffs (SURVEY.md §8f-4; src/cutoffs.jl:174-253)
# ---------------------------------------------------------------------------------------------------
def test_two_point_cutoff_literals_through_abi():
    """test/interactions.jl:1574-1635: LJ (sigma 0.3, eps 0.2) at r = 0.7 nm, dist_cutoff 0.8, dist_activation 0.6,
    evaluated by the CUDA kernels; exactly zero beyond the cutoff; unchanged below the activation distance."""
    lit = [(mb.CubicSplineCutoff(0.6, 0.8), -0.06201171875, -0.00312500000),
           (mb.PolynomialCutoff(0.6, 0.8), -0.06716652806, -0.00246320097)]
    for cut, f_ref, e_ref in lit:
        for dtype, tol in ((np.float64, 1e-9), (np.float32, 2e-7)):
            atoms = mb.atoms_from_arrays([10, 10], [1.0, 1.0], [0.3, 0.3], [0.2, 0.2], dtype)
            def pair(r):
                s = mb.System(atoms=atoms, coords=np.array([[1.0, 1, 1], [1.0 + r, 1, 1]]), boundary=mb.CubicBoundary(5.0),
                              pairwise_inters=(mb.LennardJones(cutoff=cut),), dtype=dtype)
                out = mb.forces(s)[1, 0], mb.potential_energy(s)
                s.close()
                return out
            f, e = pair(0.7)
            assert abs(f - f_ref) < tol and abs(e - e_ref) < tol, (cut, dtype, f, e)
            f, e = pair(0.85)
            assert f == 0.0 and e == 0.0
            f, e = pair(0.5)
            f0, e0 = -24 * 0.2 / 0.5 * (2 * 0.6 ** 12 - 0.6 ** 6), 4 * 0.2 * (0.6 ** 12 - 0.6 ** 6)  # plain LJ, sigma/r = 0.6
            assert abs(f + f0) < 50 * tol and abs(e - e0) < 50 * tol
    with pytest.raises(ValueError):
        mb.CubicSplineCutoff(0.8, 0.6)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("cut", ["cubic_spline", "polynomial"])
def test_two_point_cutoffs_brick_and_allpairs(dtype, cut):
    """CubicSpline / Polynomial cutoffs on LJ + Coulomb through both kernels vs the oracle
    (exercised by the reference in test/simulation.jl:565-572, test/energy_conservation.jl:21-26)."""
    mcut = {"cubic_spline": mb.CubicSplineCutoff, "polynomial": mb.PolynomialCutoff}[cut](0.8, 1.0)
    ocut = {"cubic_spline": o.CUT_CUBIC_SPLINE, "polynomial": o.CUT_POLYNOMIAL}[cut]
    mi = (mb.LennardJones(cutoff=mcut, weight_special=0.5, use_neighbors=True),
          mb.Coulomb(cutoff=mcut, weight_special=0.8333, use_neighbors=True))
    oi = [o.Inter(o.LJ, ocut, 1.0, r_act=0.8, weight_special=0.5, use_neighbors=True),
          o.Inter(o.COULOMB, ocut, 1.0, r_act=0.8, weight_special=0.8333, use_neighbors=True)]
    sd = H.molecular_system(1000, [5.1, 5.4, 5.8], seed=5)
    _check(sd, mi, oi, dtype, r_list=1.1, expect_path=1, label=f"molecular brick {cut}")
    sd = H.molecular_system(150, [3.0, 3.2, 3.4], seed=11)
    _check(sd, mi, oi, dtype, r_list=1.25, expect_path=0, label=f"molecular all-pairs {cut}")  # 3.0 nm < 2.5 r_list: no-list kernel
    sd = H.lj_fluid(9, seed=42, dtype=np.float64)
    _check(sd, (mb.LennardJones(cutoff=mcut, use_neighbors=True),), [o.Inter(o.LJ, ocut, 1.0, r_act=0.8, use_neighbors=True)],
           dtype, r_list=1.1, expect_path=1, label=f"LJ fluid {cut} (uniform)")


# ---------------------------------------------------------------------------------------------------
# step-adjacent pieces (SURVEY.md §8f-2)
# ---------------------------------------------------------------------------------------------------
def test_random_velocities_and_kinetic_tensor(golden_6mrr):
    """random_velocities! on the device: moments as test/basic.jl:53-72 checks them (statistical parity, SURVEY §8c);
    kinetic energy tensor (src/energy.jl:56-70) against numpy."""
    g = golden_6mrr
    atoms = mb.atoms_from_arrays(g["mass"], g["charge"], g["sigma"], g["eps"], np.float64)
    s = mb.System(atoms=atoms, coords=g["coords"], boundary=mb.CubicBoundary(*g["box"]), velocities=g["velocities_300K"],
                  pairwise_inters=(mb.LennardJones(cutoff=mb.DistanceCutoff(1.0), use_neighbors=True),),
                  neighbor_finder=mb.GPUNeighborFinder(dist_cutoff=1.2), dtype=np.float64)
    K = mb.kinetic_energy_tensor(s)
    K_ref = 0.5 * np.einsum("i,ia,ib->ab", g["mass"], g["velocities_300K"], g["velocities_300K"])
    assert np.abs(K - K_ref).max() < 1e-9 * np.abs(K_ref).max()
    assert abs(np.trace(K) - 65521.87288132431) < 1.5e-8 * 65521.87288132431  # test/protein.jl:284
    v = mb.random_velocities(s, 300.0, rng=np.random.default_rng(5))
    sd_ref = np.sqrt(mb.BOLTZMANN_K * 300.0 / g["mass"])
    z = v / sd_ref[:, None]
    n = z.size
    print(f"[random_velocities] mean={z.mean():.4f} var={z.var():.4f} kurt={np.mean(z ** 4):.3f} n={n}")
    assert abs(z.mean()) < 4 / np.sqrt(n) and abs(z.var() - 1) < 4 * np.sqrt(2 / n) and abs(np.mean(z ** 4) - 3) < 0.1
    assert abs(np.corrcoef(z[:, 0], z[:, 1])[0, 1]) < 4 / np.sqrt(len(z))
    s.velocities[...] = v
    assert abs(mb.temperature(s) - 300.0) < 6.0
    v2 = mb.random_velocities(s, 300.0, rng=np.random.default_rng(5))
    assert np.array_equal(v, v2)  # same rng state -> same stream
    s.close()


# ---------------------------------------------------------------------------------------------------
# TriclinicBoundary (SURVEY.md §8f-4; src/spatial.jl:528-551, :584-600)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_triclinic_boundary(dtype):
    """test/gpu_consistency.jl:287-337: 50 atoms in the box (2,0,0), (0.1,2,0), (0.2,0.3,2), LJ sigma 0.3, eps 1, cutoff 0.8;
    forces and energy against the numpy oracle (the reference compares its GPU and CPU paths at rtol 1e-8); then a short
    VelocityVerlet run: wrapped output, momentum conserved, trajectory against the oracle's arithmetic."""
    from oracle import triclinic as tr
    bv = np.array([[2.0, 0.0, 0.0], [0.1, 2.0, 0.0], [0.2, 0.3, 2.0]])
    rng = np.random.default_rng(42)
    n = 50
    # rejection sampling keeps pairs apart (the reference's rand()*1.5 coordinates hold overlaps with forces ~1e12; the
    # comparison is relative either way)
    pts = []
    t = tr.Triclinic(bv)
    while len(pts) < n:
        c = rng.random(3) * 1.9
        if all(np.linalg.norm(t.vector(p, c)) > 0.27 for p in pts):
            pts.append(c)
    x = np.array(pts)
    sigma, eps = np.full(n, 0.3), np.ones(n)
    f_ref, e_ref, vir_ref = tr.forces_energy(t, x, sigma, eps, r_cut=0.8)
    atoms = mb.atoms_from_arrays(np.ones(n), np.zeros(n), sigma, eps, dtype)
    s = mb.System(atoms=atoms, coords=x.astype(dtype), boundary=mb.TriclinicBoundary(*bv),
                  pairwise_inters=(mb.LennardJones(cutoff=mb.DistanceCutoff(0.8), use_neighbors=True),),
                  neighbor_finder=mb.GPUNeighborFinder(dist_cutoff=0.8), dtype=dtype)
    f = mb.forces(s)
    e = mb.potential_energy(s)
    f2, vir = mb.forces_virial(s)
    tol = 1e-8 if dtype == np.float64 else 2e-5
    fmax = np.abs(f_ref).max()
    print(f"[triclinic] dtype={np.dtype(dtype).name} max|dF|={np.abs(f - f_ref).max():.3e} (max|F|={fmax:.3e}) dE={e - e_ref:.3e} path={s.stats()['path']}")
    assert s.stats()["path"] == 0
    assert np.abs(f - f_ref).max() <= tol * fmax + 1e-10
    assert abs(e - e_ref) <= tol * abs(e_ref) + 1e-10
    assert np.abs(vir - vir_ref).max() <= 10 * tol * np.abs(vir_ref).max() + 1e-9
    # dynamics: velocity Verlet in the triclinic box (test/basic.jl:236-262 does the same with free particles)
    v0 = rng.normal(0, 0.3, (n, 3))
    v0 -= v0.mean(0)
    s.velocities[...] = v0.astype(dtype)
    mb.simulate(s, mb.VelocityVerlet(dt=0.001, remove_CM_motion=0), 50)
    xw = np.array([t.wrap(v) for v in s.coords.astype(np.float64)])
    assert np.abs(xw - s.coords).max() < (1e-12 if dtype == np.float64 else 1e-5)  # returned coordinates are wrapped
    p = s.velocities.astype(np.float64).sum(0)
    assert np.abs(p).max() < (1e-9 if dtype == np.float64 else 1e-3)
    if dtype == np.float64:  # the same 50 steps in numpy with the oracle's forces
        xr, vr = x.copy(), v0.copy()
        fr = f_ref
        for _ in range(50):
            vr = vr + fr * 0.0005
            xr = np.array([t.wrap(q) for q in xr + vr * 0.001])
            fr, _, _ = tr.forces_energy(t, xr, sigma, eps, r_cut=0.8)
            vr = vr + fr * 0.0005
        d = np.array([t.vector(a, b) for a, b in zip(xr, s.coords)])
        print(f"[triclinic] 50 VV steps: max|dx|={np.abs(d).max():.3e} max|dv|={np.abs(vr - s.velocities).max():.3e}")
        assert np.abs(d).max() < 1e-9 and np.abs(vr - s.velocities).max() < 1e-8
    s.close()
    # the engine refuses what it does not implement for such a box
    with pytest.raises(ValueError):
        mb.TriclinicBoundary([2.0, 0.1, 0.0], [0.0, 2.0, 0.0], [0.0, 0.0, 2.0])


# ---------------------------------------------------------------------------------------------------
# energy conservation, the reference's protocol (test/energy_conservation.jl:9-75)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cut", ["distance", "shifted_potential", "shifted_force", "cubic_spline"])
def test_energy_conservation_reference_protocol(cut):
    """2 000 atoms (m 40, sigma 0.05, eps 0.2) at 1 K in a 5 nm box, LJ with dist_cutoff 3.0 nm, VelocityVerlet dt 1 fs without
    CM removal, Float64: max |E(t) - E0| over 10 000 steps (sampled every 100) < 5e-4 kJ/mol, final coordinates inside the box."""
    n, L, rc = 2000, 5.0, 3.0
    rng = np.random.default_rng(11)
    pts = np.empty((0, 3))
    while len(pts) < n:  # place_atoms(n, boundary; min_dist = 0.1) (src/setup.jl:23-60): rejection sampling, in batches
        c = rng.random((4 * n, 3)) * L
        for q in c:
            d = pts - q
            d -= L * np.round(d / L)
            if len(pts) == 0 or (np.einsum("ij,ij->i", d, d) > 0.01).all():
                pts = np.vstack([pts, q])
                if len(pts) == n:
                    break
    cutoff = {"distance": mb.DistanceCutoff(rc), "shifted_potential": mb.ShiftedPotentialCutoff(rc),
              "shifted_force": mb.ShiftedForceCutoff(rc), "cubic_spline": mb.CubicSplineCutoff(rc, rc + 0.5)}[cut]
    mass = np.full(n, 40.0)
    atoms = mb.atoms_from_arrays(mass, np.zeros(n), np.full(n, 0.05), np.full(n, 0.2), np.float64)
    v = rng.normal(0.0, np.sqrt(mb.BOLTZMANN_K * 1.0 / 40.0), (n, 3))
    s = mb.System(atoms=atoms, coords=pts.copy(), boundary=mb.CubicBoundary(L), velocities=v,
                  pairwise_inters=(mb.LennardJones(cutoff=cutoff, use_neighbors=True),),
                  neighbor_finder=mb.GPUNeighborFinder(dist_cutoff=rc + (0.5 if cut == "cubic_spline" else 0.0)), dtype=np.float64)
    sim = mb.VelocityVerlet(dt=0.001, remove_CM_motion=0)
    e0 = mb.potential_energy(s) + mb.kinetic_energy(s)
    worst = 0.0
    for k in range(100):
        mb.simulate(s, sim, 100, init_step=100 * k)
        worst = max(worst, abs(mb.potential_energy(s) + mb.kinetic_energy(s) - e0))
    print(f"[energy conservation, {cut}] path={s.stats()['path']} E0={e0:.6f} max|E-E0| over 10000 steps = {worst:.3e} kJ/mol (bar 5e-4)")
    assert worst < 5e-4
    assert (s.coords >= 0).all() and (s.coords < L).all()
    s.close()
