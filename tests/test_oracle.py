"""CPU tests: pin the oracle against the reference's own known answers and golden vectors
(SURVEY.md §4 / §8c). No GPU needed."""
import numpy as np
import pytest

from oracle import oracle as o
import mbhelpers as H


def _pair(inter, r, q=0.0, dtype=np.float64, sig=0.3, eps=0.2, box=5.0):
    s = o.OracleSystem(box=[box] * 3, mass=[10, 10], charge=[q, q], sigma=[sig, sig], eps=[eps, eps], inters=[inter],
                       dtype=dtype)
    x = np.array([[1.0, 1.0, 1.0], [1.0 + r, 1.0, 1.0]])
    f, pe, _ = s.forces_allpairs(x, n_threads=1)
    return f[1, 0], pe  # +x force on atom j = F (positive = repulsive)


def test_mic_and_wrap_known_answers():
    # test/basic.jl:2-38
    assert o.vector_1D(4.0, 6.0, 10.0) == 2.0
    assert o.vector_1D(1.0, 9.0, 10.0) == -2.0
    assert o.wrap_coord_1D(-2.0, 10.0) == 8.0
    assert o.wrap_coord_1D(12.0, 10.0) == 2.0
    box = (10.0, 5.0, 3.5)
    v = [o.vector_1D(a, b, L) for a, b, L in zip((4.0, 1.0, 1.0), (6.0, 4.0, 3.0), box)]
    assert v == [2.0, -2.0, -1.5]


def test_lj_pair_known_answers():
    # test/interactions.jl:61-82 (sigma 0.3, eps 0.2)
    lj = o.Inter(o.LJ)
    f, e = _pair(lj, 0.3)
    assert abs(f - 16.0) < 1e-9 and abs(e - 0.0) < 1e-9
    f, e = _pair(lj, 0.4)
    assert abs(f - (-1.375509739)) < 1e-9 and abs(e - (-0.1170417309)) < 1e-9


def test_coulomb_pair_known_answers():
    # test/interactions.jl:374-395 (q = 1, 1), atol 1e-5
    c = o.Inter(o.COULOMB)
    f, e = _pair(c, 0.3, q=1.0)
    assert abs(f - 1543.727311) < 1e-5 and abs(e - 463.1181933) < 1e-5
    f, e = _pair(c, 0.4, q=1.0)
    assert abs(f - 868.3466125) < 1e-5 and abs(e - 347.338645) < 1e-5


def test_mixing_rules():
    # test/interactions.jl:15-21: Lorentz sigma of (0.2, 0.3) = 0.25; geometric eps of (0.1, 0.2)
    s = o.OracleSystem(box=[5.0] * 3, mass=[1, 1], charge=[0, 0], sigma=[0.2, 0.3], eps=[0.1, 0.2],
                       inters=[o.Inter(o.LJ)])
    x = np.array([[1.0, 1, 1], [1.25, 1, 1]])  # r = sigma_mixed -> E = 0
    _, pe, _ = s.forces_allpairs(x, n_threads=1)
    assert abs(pe) < 1e-12
    x = np.array([[1.0, 1, 1], [1.0 + 0.25 * 2 ** (1 / 6), 1, 1]])  # minimum: E = -eps_mixed
    _, pe, _ = s.forces_allpairs(x, n_threads=1)
    assert abs(pe + 0.14142135623730953) < 1e-12


def test_crf_behaviour():
    # test/interactions.jl:506-660: zero beyond cutoff; special pairs = weighted plain Coulomb
    crf = o.Inter(o.CRF, o.CUT_DISTANCE, 1.0, weight_special=0.5, use_neighbors=True)
    f, e = _pair(crf, 1.2, q=1.0)
    assert f == 0.0 and e == 0.0
    s = o.OracleSystem(box=[5.0] * 3, mass=[1, 1], charge=[1.0, 1.0], sigma=[0, 0], eps=[0, 0], inters=[crf],
                       special_pairs=np.array([[0, 1]]))
    x = np.array([[1.0, 1, 1], [1.4, 1, 1]])
    f, pe, _ = s.forces_allpairs(x, n_threads=1)
    assert abs(f[1, 0] - 0.5 * 868.34661025) < 1e-6 and abs(pe - 0.5 * 347.3386441) < 1e-6
    # eps = inf: k_rf = 1/(2 rc^3)
    crf_inf = o.Inter(o.CRF, o.CUT_DISTANCE, 1.0, solvent_dielectric=float("inf"))
    f, e = _pair(crf_inf, 0.5, q=1.0)
    ke = o.COULOMB_CONST
    assert abs(f - ke * (1 / 0.25 - 2 * 0.5 * 0.5)) < 1e-9
    assert abs(e - ke * (1 / 0.5 + 0.5 * 0.25 - 1.5)) < 1e-9


def test_cutoff_algebra():
    # test/interactions.jl:1574-1635 relations: shifted potential is continuous at rc, shifted force has F(rc)=0
    for kind in (o.LJ, o.COULOMB):
        q = 1.0 if kind == o.COULOMB else 0.0
        plain = o.Inter(kind, o.CUT_DISTANCE, 0.8)
        sp = o.Inter(kind, o.CUT_SHIFTED_POTENTIAL, 0.8)
        sf = o.Inter(kind, o.CUT_SHIFTED_FORCE, 0.8)
        f0, e0 = _pair(plain, 0.5, q)
        f1, e1 = _pair(sp, 0.5, q)
        f2, e2 = _pair(sf, 0.5, q)
        fc, ec = _pair(plain, 0.8, q)
        assert abs(f1 - f0) < 1e-12 and abs(e1 - (e0 - ec)) < 1e-12
        assert abs(f2 - (f0 - fc)) < 1e-12 and abs(e2 - (e0 + (0.5 - 0.8) * fc - ec)) < 1e-12
        fe, ee = _pair(sf, 0.8 - 1e-12, q)
        assert abs(fe) < 1e-6 and abs(ee) < 1e-9
        assert _pair(sf, 0.81, q) == (0.0, 0.0)


def test_6mrr_pair_count(golden_6mrr):
    # test/basic.jl:592-593: exactly 4 602 420 eligible pairs within 1.2 nm
    g = golden_6mrr
    s = o.OracleSystem(box=g["box"], mass=g["mass"], charge=g["charge"], sigma=g["sigma"], eps=g["eps"],
                       inters=[o.Inter(o.LJ, o.CUT_DISTANCE, 1.0, use_neighbors=True)], excluded_pairs=g["excluded"],
                       special_pairs=g["special"])
    x = g["coords"] - np.floor(g["coords"] / g["box"]) * g["box"]
    nl = s.neighbor_list(x, 1.2)
    assert len(nl) == 4602420
    assert int(nl[:, 2].sum()) == len(g["special"])


@pytest.mark.parametrize("name", ["lj_only", "coul_only"])
def test_6mrr_openmm_golden(golden_6mrr, name):
    # test/protein.jl:206-276: max |dF| < 1e-7 kJ/mol/nm, |dE| < 1e-5 kJ/mol vs OpenMM Reference platform
    g = golden_6mrr
    if name == "lj_only":
        inter = o.Inter(o.LJ, o.CUT_DISTANCE, 1.0, weight_special=float(g["lj14scale"]), use_neighbors=True)
    else:
        inter = o.Inter(o.CRF, o.CUT_DISTANCE, 1.0, weight_special=float(g["coulomb14scale"]), use_neighbors=True)
    s = o.OracleSystem(box=g["box"], mass=g["mass"], charge=g["charge"], sigma=g["sigma"], eps=g["eps"], inters=[inter],
                       excluded_pairs=g["excluded"], special_pairs=g["special"])
    x = g["coords"] - np.floor(g["coords"] / g["box"]) * g["box"]
    f, pe, _ = s.forces_allpairs(x)
    if name == "lj_only":
        pe += o.lj_dispersion_correction_energy(g["sigma"], g["eps"], g["box"], 1.0)
    assert np.linalg.norm(f[g["openmm_sample"]] - g[f"forces_{name}"], axis=1).max() < 1e-7
    assert abs(pe - float(g[f"energy_{name}"])) < 1e-5
    # neighbour-list path of the oracle agrees with brute force
    nl = s.neighbor_list(x, 1.0 + 0.2)
    f2, pe2, _ = s.forces_nl(x, nl)
    assert np.abs(f2 - f).max() < 1e-8
    if name == "lj_only":
        pe2 += o.lj_dispersion_correction_energy(g["sigma"], g["eps"], g["box"], 1.0)
    assert abs(pe2 - pe) < 1e-7


def test_6mrr_kinetic_energy_and_temperature(golden_6mrr):
    # test/protein.jl:284-286
    g = golden_6mrr
    ke = o.kinetic_energy(g["mass"], g["velocities_300K"])
    # the reference uses isapprox (rtol = sqrt(eps) = 1.5e-8)
    assert abs(ke - 65521.87288132431) < 1.5e-8 * 65521.87288132431
    assert abs(o.temperature(g["mass"], g["velocities_300K"]) - 329.3202932884933) < 1.5e-8 * 329.3202932884933


def test_vv_oracle_conserves_energy_and_momentum():
    sd = H.lj_fluid(4, seed=3, dtype=np.float64)  # 256 atoms
    inter = o.Inter(o.LJ, o.CUT_SHIFTED_FORCE, 1.0, use_neighbors=True)
    s = H.make_oracle(sd, [inter])
    x0, v0 = sd["coords"], sd["velocities"]
    _, pe0, _ = s.forces_allpairs(x0)
    e0 = pe0 + o.kinetic_energy(sd["mass"], v0)
    x1, v1, pe1 = s.simulate_vv(x0, v0, 0.002, 200, remove_cm_every=1, r_list=1.2, nl_every=10)
    e1 = pe1 + o.kinetic_energy(sd["mass"], v1)
    assert abs(e1 - e0) < 5e-3 * abs(e0) / 100 + 0.05
    assert np.abs((sd["mass"][:, None] * v1).sum(0)).max() < 1e-9
    assert (x1 >= 0).all() and (x1 < sd["box"]).all()
    # f32 instantiation tracks f64
    s32 = H.make_oracle(sd, [inter], dtype=np.float32)
    x2, v2, _ = s32.simulate_vv(x0, v0, 0.002, 20, r_list=1.2)
    x3, v3, _ = s.simulate_vv(x0, v0, 0.002, 20, r_list=1.2)
    d = x2.astype(np.float64) - x3
    d -= sd["box"] * np.round(d / sd["box"])
    assert np.abs(d).max() < 1e-4


@pytest.mark.parametrize("name,idx,par", [("bond_only", "bond_idx", "bond_par"), ("angle_only", "angle_idx", "angle_par"),
                                          ("proptor_only", "proper_idx", "proper_par"),
                                          ("improptor_only", "improper_idx", "improper_par")])
def test_6mrr_bonded_openmm_golden(golden_6mrr, name, idx, par):
    # test/protein.jl:206-276: bonded terms vs OpenMM (energies 164735.97 / 2839.82 / 2892.48 / 128.24 kJ/mol)
    from oracle import bonded as bd
    g = golden_6mrr
    fn = {"bond_only": bd.bond_forces, "angle_only": bd.angle_forces}.get(name, bd.torsion_forces)
    f, e = fn(g["coords"], g["box"], g[idx], g[par])
    assert np.linalg.norm(f[g["openmm_sample"]] - g[f"forces_{name}"], axis=1).max() < 1e-7
    assert abs(e - float(g[f"energy_{name}"])) < 1e-5


def test_6mrr_all_cut_openmm_golden(golden_6mrr):
    # the whole :cutoff system: LJ + CRF + bonded (+ LJ dispersion correction in the energy), E = 41763.84577241427
    g = golden_6mrr
    orc, sd = H.sixmrr_oracle(g)
    f, e, _ = orc.forces_allpairs(sd["coords"])
    fb, eb = H.bonded_forces_oracle(g, sd["coords"])
    e += eb + o.lj_dispersion_correction_energy(g["sigma"], g["eps"], g["box"], 1.0)
    assert np.linalg.norm((f + fb)[g["openmm_sample"]] - g["forces_all_cut"], axis=1).max() < 1e-7
    assert abs(e - float(g["energy_all_cut"])) < 1e-5


def test_6mrr_all_pme_openmm_golden(golden_6mrr):
    """SURVEY.md §8(f)-3 oracle pin: the :pme system = LJ + CoulombEwald real space (C oracle) + bonded + EwaldExclusion
    over excluded-or-special pairs + PME reciprocal space with self/background terms (oracle/pme.py), against OpenMM's
    forces_all_pme_exact / energy_all_pme_exact with the reference's own tolerances (test/protein.jl:267, :274)."""
    from oracle import pme
    g = golden_6mrr
    sd = H.sixmrr_description(g)
    alpha = pme.pme_alpha(1.0)
    assert pme.pme_mesh_dims(g["box"], alpha) == (46, 46, 51)
    inters = [o.Inter(o.LJ, o.CUT_DISTANCE, 1.0, weight_special=float(g["lj14scale"]), use_neighbors=True),
              o.Inter(o.EWALD_REAL, o.CUT_DISTANCE, 1.0, weight_special=float(g["coulomb14scale"]), ewald_alpha=alpha,
                      use_neighbors=True)]
    orc = H.make_oracle(sd, inters, dtype=np.float64)
    f, e, _ = orc.forces_allpairs(sd["coords"])
    fb, eb = H.bonded_forces_oracle(g, sd["coords"])
    fr, er, _ = pme.pme_reciprocal(sd["coords"], g["charge"], g["box"], r_cut=1.0, error_tol=0.0005, order=5)
    fx, ex = pme.ewald_exclusion(sd["coords"], g["charge"], g["box"], np.concatenate([g["excluded"], g["special"]]))
    e_tot = e + eb + er + ex + o.lj_dispersion_correction_energy(g["sigma"], g["eps"], g["box"], 1.0)
    assert np.linalg.norm((f + fb + fr + fx)[g["openmm_sample"]] - g["forces_all_pme_exact"], axis=1).max() < 1e-7
    assert abs(e_tot - float(g["energy_all_pme_exact"])) < 1e-5


def test_6mrr_all_pme_approx_erfc_openmm_golden(golden_6mrr):
    """The reference's DEFAULT CoulombEwald (approximate_erfc=true, coulomb.jl:1331, calc_erfc :1384-1393) against
    OpenMM's non-exact goldens forces_all_pme / energy_all_pme with the reference's tolerances for that case
    (test/protein.jl:267, :274: 1e-3 kJ/mol/nm, 0.2 kJ/mol)."""
    from oracle import pme
    g = golden_6mrr
    sd = H.sixmrr_description(g)
    alpha = pme.pme_alpha(1.0)
    inters = [o.Inter(o.LJ, o.CUT_DISTANCE, 1.0, weight_special=float(g["lj14scale"]), use_neighbors=True),
              o.Inter(o.EWALD_REAL, o.CUT_DISTANCE, 1.0, weight_special=float(g["coulomb14scale"]), ewald_alpha=alpha,
                      use_neighbors=True, approx_erfc=True)]
    orc = H.make_oracle(sd, inters, dtype=np.float64)
    f, e, _ = orc.forces_allpairs(sd["coords"])
    fb, eb = H.bonded_forces_oracle(g, sd["coords"])
    fr, er, _ = pme.pme_reciprocal(sd["coords"], g["charge"], g["box"], r_cut=1.0, error_tol=0.0005, order=5)
    fx, ex = pme.ewald_exclusion(sd["coords"], g["charge"], g["box"], np.concatenate([g["excluded"], g["special"]]))
    e_tot = e + eb + er + ex + o.lj_dispersion_correction_energy(g["sigma"], g["eps"], g["box"], 1.0)
    df = np.linalg.norm((f + fb + fr + fx)[g["openmm_sample"]] - g["forces_all_pme"], axis=1).max()
    de = abs(e_tot - float(g["energy_all_pme"]))
    print("approx erfc vs all_pme: max|dF| =", df, "dE =", de)
    assert df < 1e-3 and de < 0.2
    # (the reference ships byte-identical all_pme / all_pme_exact files: the looser tolerance IS the polynomial's error,
    # measured here 4.6e-4 kJ/mol/nm and 0.12 kJ/mol; the exact variant must not pass the tight bar by accident)
    assert df > 1e-7


def test_6mrr_vv_100steps_openmm_trajectory(golden_6mrr):
    """Oracle pin of the WHOLE step loop: 100 VelocityVerlet steps (dt 0.5 fs) of the :pme system from velocities_300K
    against OpenMM's coordinates_100steps / velocities_100steps with the reference's bars (test/protein.jl:277-299:
    1e-10 nm, 1e-7 nm/ps)."""
    g = golden_6mrr
    sd = H.sixmrr_description(g)
    x, v = H.oracle_vv_pme(g, sd["coords"], g["velocities_300K"], 0.0005, 100)
    box = g["box"]
    x_ref = g["coordinates_100steps"] - np.floor(g["coordinates_100steps"] / box) * box
    d = x[g["openmm_sample"]] - x_ref
    d -= box * np.round(d / box)
    dx, dv = np.linalg.norm(d, axis=1).max(), np.linalg.norm(v[g["openmm_sample"]] - g["velocities_100steps"], axis=1).max()
    print("oracle VV 100 steps vs OpenMM: dx =", dx, "dv =", dv)
    assert dx < 1e-10 and dv < 1e-7


def test_cutoff_literals_all_six():
    """test/interactions.jl:1574-1635: LJ (sigma 0.3, eps 0.2) at r = 0.7 nm under the six cutoffs (dist_cut 0.8,
    dist_act 0.6), and exactly zero at r = 1.0 / 0.95 nm. CubicSpline / Polynomial (SURVEY.md §8f-4) exist in the
    oracle only so far."""
    lit = [(o.CUT_NONE, -0.04196301990, -0.00492640193), (o.CUT_DISTANCE, -0.04196301990, -0.00492640193),
           (o.CUT_SHIFTED_POTENTIAL, -0.04196301990, -0.00270785727), (o.CUT_SHIFTED_FORCE, -0.02537033587, -0.00104858887),
           (o.CUT_CUBIC_SPLINE, -0.06201171875, -0.00312500000), (o.CUT_POLYNOMIAL, -0.06716652806, -0.00246320097)]
    for kind, f_ref, e_ref in lit:
        s = o.OracleSystem(box=np.array([2.0, 2.0, 2.0]), mass=np.ones(2), charge=np.ones(2), sigma=np.full(2, 0.3),
                           eps=np.full(2, 0.2), inters=[o.Inter(o.LJ, kind, 0.8, r_act=0.6)])
        f, e, _ = s.forces_allpairs(np.array([[1.0, 1.0, 1.0], [1.7, 1.0, 1.0]]))
        # the reference's force(inter, dr, ...) is f with fs[i] -= f, fs[j] += f (src/force.jl:869-874)
        assert abs(f[1, 0] - f_ref) < 1e-9 and abs(f[0, 0] + f_ref) < 1e-9 and abs(e - e_ref) < 1e-9
        if kind != o.CUT_NONE:
            for xj in (2.0, 1.95):  # minimum image: r = 1.0 and 0.95 nm, both beyond the cutoff
                f, e, _ = s.forces_allpairs(np.array([[1.0, 1.0, 1.0], [xj, 1.0, 1.0]]))
                assert np.abs(f).max() < 1e-12 and abs(e) < 1e-12


def test_water3_pme_openmm_literals():
    """Second PME pin, on a non-cubic orthorhombic box (2.0 x 2.1 x 2.2 nm): three TIP3P waters, electrostatics only,
    dist_cutoff 0.9 nm — the OpenMM energy / forces the reference's "Ewald" testset holds as literals
    (test/interactions.jl:1683-1697; its tolerances: 2e-4 kJ/mol, 5e-4 kJ/mol/nm)."""
    import os
    from oracle import pme
    w = dict(np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "water3.npz")))
    rc = float(w["r_cut"])
    alpha = pme.pme_alpha(rc)
    assert pme.pme_mesh_dims(w["box"], alpha) == (18, 19, 20)
    s = o.OracleSystem(box=w["box"], mass=w["mass"], charge=w["charge"], sigma=w["sigma"], eps=w["eps"],
                       inters=[o.Inter(o.EWALD_REAL, o.CUT_DISTANCE, rc, ewald_alpha=alpha, use_neighbors=True)],
                       excluded_pairs=w["excluded"], special_pairs=w["special"])
    f, e, _ = s.forces_allpairs(w["coords"])
    fr, er, _ = pme.pme_reciprocal(w["coords"], w["charge"], w["box"], r_cut=rc)
    fx, ex = pme.ewald_exclusion(w["coords"], w["charge"], w["box"], w["excluded"], r_cut=rc)
    assert np.linalg.norm(f + fr + fx - w["forces_pme"], axis=1).max() < 1e-7  # reference: 5e-4
    assert abs(e + er + ex - float(w["energy_pme"])) < 1e-8                   # reference: 2e-4


def test_triclinic_oracle_pins():
    """oracle/triclinic.py against the reference's own checks: basis-vector literals of the lengths + angles constructor
    (test/basic.jl:130-135), wrap_coords leaves in-box coordinates alone (:219), the approximate minimum image equals the exact
    27-image search up to half the smallest height (:221-234)."""
    from oracle import triclinic as tr
    bv = tr.basis_from_lengths_angles([2.2, 2.0, 1.8], np.deg2rad([50.0, 40.0, 60.0]))
    lit = np.array([[2.2, 0.0, 0.0], [1.0, 1.7320508, 0.0], [1.37888, 0.5399122, 1.0233204]])
    assert np.abs(bv - lit).max() < 1e-6
    t = tr.Triclinic(bv)
    rng = np.random.default_rng(7)
    x = rng.random((1000, 3)) @ bv  # fractional coordinates in [0, 1): inside the box
    assert all(np.array_equal(t.wrap(v), v) or np.abs(t.wrap(v) - v).max() < 1e-12 for v in x)
    lim = min(bv[0, 0], bv[1, 1], bv[2, 2]) / 2
    n_checked = 0
    for i in range(999):
        de = t.vector_exact(x[i], x[i + 1])
        if np.linalg.norm(de) <= lim:
            n_checked += 1
            assert np.allclose(de, t.vector(x[i], x[i + 1]), atol=1e-12)
    assert n_checked > 100
    # out-of-box coordinates come back inside, displaced by lattice vectors only
    y = x + rng.integers(-2, 3, (1000, 3)) @ bv
    w = np.array([t.wrap(v) for v in y])
    assert np.abs(w - x).max() < 1e-9
    with pytest.raises(ValueError):
        tr.Triclinic([[2.0, 0.1, 0.0], [0.0, 2.0, 0.0], [0.0, 0.0, 2.0]])
