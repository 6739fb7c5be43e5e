"""Generate tests/golden/*.npz from the reference's own data files.

Reads the `data/` directory of a Molly.jl checkout and writes small fixtures: the
6mrr system (per-atom parameters, exclusions, 1-4 specials derived by
oracle/ffreader.py) and the OpenMM golden forces/energies the reference's
test/protein.jl:206-276 compares against, plus per-pair literals. The per-atom
OpenMM arrays (forces, the state after 100 steps) are kept for a fixed, seeded
sample of OPENMM_SAMPLE atoms, listed in `openmm_sample`, so that the fixture
stays under 1 MB; the energies cover the whole system.
Usage: python oracle/make_golden.py <Molly.jl>/data
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ffreader as fr  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
OPENMM_SAMPLE = 1024


def main(ref):
    os.makedirs(OUT, exist_ok=True)
    ff = fr.read_force_field(f"{ref}/force_fields/ff99SBildn.xml", f"{ref}/force_fields/tip3p_standard.xml")
    atoms, box = fr.read_pdb(f"{ref}/6mrr_equil.pdb")
    top = fr.build_topology(atoms, ff)
    coords = np.array([a.xyz for a in atoms], np.float64)
    amber = f"{ref}/openmm_6mrr/amber"
    out = dict(
        box=box, coords=coords, mass=top["mass"], charge=top["charge"], sigma=top["sigma"], eps=top["eps"],
        excluded=top["excluded"], special=top["special"],
        lj14scale=np.float64(ff.lj14scale), coulomb14scale=np.float64(ff.coulomb14scale),
        velocities_300K=np.loadtxt(f"{ref}/openmm_6mrr/velocities_300K.txt"),
    )
    for key in ("bond_idx", "bond_par", "angle_idx", "angle_par", "proper_idx", "proper_par", "improper_idx", "improper_par"):
        out[key] = top[key]
    for name in ("lj_only", "coul_only", "bond_only", "angle_only", "proptor_only", "improptor_only", "all_cut",
                 "all_pme_exact", "all_pme"):
        out[f"forces_{name}"] = np.loadtxt(f"{amber}/forces_{name}.txt")
        out[f"energy_{name}"] = np.float64(open(f"{amber}/energy_{name}.txt").read())
    # 100 VelocityVerlet steps of the :pme system from velocities_300K (test/protein.jl:277-299: 1e-10 nm, 1e-7 nm/ps)
    out["coordinates_100steps"] = np.loadtxt(f"{amber}/coordinates_100steps.txt")
    out["velocities_100steps"] = np.loadtxt(f"{amber}/velocities_100steps.txt")
    sample = np.sort(np.random.default_rng(0).choice(len(coords), OPENMM_SAMPLE, replace=False)).astype(np.int32)
    for key in [k for k in out if k.startswith("forces_")] + ["coordinates_100steps", "velocities_100steps"]:
        out[key] = out[key][sample]
    out["openmm_sample"] = sample
    np.savez_compressed(os.path.join(OUT, "6mrr.npz"), **out)
    print("wrote", os.path.join(OUT, "6mrr.npz"), os.path.getsize(os.path.join(OUT, "6mrr.npz")) / 1e6, "MB")
    water3(ref)


def water3(ref):
    """Three TIP3P waters in a 2.0 x 2.1 x 2.2 nm box (data/water_3mol_cubic.pdb), electrostatics only, dist_cutoff 0.9:
    the OpenMM energies / forces the reference's "Ewald" testset holds as literals (test/interactions.jl:1638-1650 for
    :ewald, :1683-1697 for :pme; tolerances there: 2e-4 kJ/mol, 5e-4 kJ/mol/nm)."""
    ff = fr.read_force_field(f"{ref}/force_fields/tip3p_standard.xml")
    atoms, box = fr.read_pdb(f"{ref}/water_3mol_cubic.pdb")
    top = fr.build_topology(atoms, ff)
    f_pme = np.array([
        [-72.57603365363543, 5.648072796188359, 101.40821248959712], [17.558243038254187, 4.075128117683555, -37.70060863840432],
        [30.881405092779705, -12.047169393065978, -32.137723916688024], [-7.789998310481266, -14.185855369417702, -8.35080870148926],
        [2.3519124244832277, 7.264285806008946, 4.431212066763443], [7.085282096874462, 8.530075688459654, 5.32165402278671],
        [-97.20750157586099, 14.85484666061426, 63.32187921636768], [48.50069206640984, 4.544995194749845, -21.497171353580004],
        [71.21703702929426, -18.67010037709364, -74.8362731945127]])
    f_ewald = np.array([
        [-72.48152122617766, 5.6452093242736225, 101.4156707298087], [17.520231752234416, 4.071455080698861, -37.701631053185295],
        [30.858153727989023, -12.062341554089436, -32.14366235405959], [-7.936279084919704, -14.215671548792962, -8.295642564943837],
        [2.4095151618606145, 7.275822557366837, 4.433671630065675], [7.141770437453555, 8.540348761741292, 5.30999589638612],
        [-97.27674352036883, 14.881678867954054, 63.35431221886955], [48.485910228223275, 4.532352998517133, -21.51089738652309],
        [71.2789625237053, -18.668854487669485, -74.8618171164182]])
    np.savez_compressed(os.path.join(OUT, "water3.npz"), box=box, coords=np.array([a.xyz for a in atoms], np.float64),
                        charge=top["charge"], mass=top["mass"], sigma=top["sigma"], eps=top["eps"], excluded=top["excluded"],
                        special=top["special"], r_cut=np.float64(0.9), forces_pme=f_pme, energy_pme=np.float64(-5.460124320435284),
                        forces_ewald=f_ewald, energy_ewald=np.float64(-5.465127432466375))
    print("wrote", os.path.join(OUT, "water3.npz"))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
