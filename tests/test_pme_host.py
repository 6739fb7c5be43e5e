"""The PME device functions, run on the HOST (SURVEY.md §8(f)-3). csrc/pme.cuh writes every kernel as a thin loop over a
__host__ __device__ per-item function; tests/host/pme_host.cu compiles those functions for the CPU (nvcc, host code
only) and this test drives spread -> FFT (numpy) -> convolution -> inverse FFT -> interpolation -> exclusion with them and
compares with the numpy oracle and, end to end, with OpenMM's forces_all_pme_exact for 6mrr. What this does NOT cover is
the CUDA launch plumbing, the atomics and cuFFT (tests/test_zz_gpu_pme.py, xfail until it has run on a GPU)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import mbhelpers as H
from oracle import oracle as o
from oracle import pme

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hostlib(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("pmeh") / "libpmeh.so")
    cmd = [nvcc, "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++", "-gencode",
           "arch=compute_100a,code=sm_100a", "-o", out, os.path.join(ROOT, "tests", "host", "pme_host.cu")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    L = C.CDLL(out)
    L.pmeh_conv.restype = C.c_double
    L.pmeh_exclusion.restype = C.c_double
    return L


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def test_pme_device_functions_on_host_vs_openmm(hostlib, golden_6mrr):
    g = golden_6mrr
    sd = H.sixmrr_description(g)
    n = sd["n"]
    box = np.ascontiguousarray(g["box"], np.float64)
    alpha = pme.pme_alpha(1.0)
    K = np.array(pme.pme_mesh_dims(box, alpha), np.int32)
    bsm = [np.ascontiguousarray(m) for m in pme.bspline_moduli(5, tuple(K))]
    pos4 = np.ascontiguousarray(np.concatenate([sd["coords"], g["charge"][:, None]], 1), np.float64)
    f_div = pme.COULOMB_CONST
    # spread with the device function, compare the grid with the oracle's spreading
    grid = np.zeros((K[0], K[1], K[2], 2), np.float64)
    hostlib.pmeh_spread(n, _ptr(K), _ptr(box), _ptr(pos4), _ptr(grid))
    assert abs(grid[..., 0].sum() - g["charge"].sum()) < 1e-9 and not grid[..., 1].any()
    S = np.fft.fftn(grid[..., 0])
    cg = np.ascontiguousarray(np.stack([S.real, S.imag], -1))
    e_recip = hostlib.pmeh_conv(_ptr(K), _ptr(box), C.c_double(f_div), C.c_double(alpha), _ptr(bsm[0]), _ptr(bsm[1]), _ptr(bsm[2]), _ptr(cg))
    pot = np.fft.ifftn(cg[..., 0] + 1j * cg[..., 1]) * K.prod()  # cuFFT's inverse is unnormalised, like bfft!
    pg = np.ascontiguousarray(np.stack([pot.real, pot.imag], -1))
    f4 = np.zeros((n, 4), np.float64)
    hostlib.pmeh_interp(n, _ptr(K), _ptr(box), _ptr(pos4), _ptr(pg), _ptr(f4))
    fr_ref, er_ref, info = pme.pme_reciprocal(sd["coords"], g["charge"], box)
    assert np.abs(f4[:, :3] - fr_ref).max() < 1e-9 * max(1.0, np.abs(fr_ref).max())
    assert abs(e_recip - info["e_recip"]) < 1e-9 * abs(info["e_recip"])
    # exclusion correction
    pairs = np.ascontiguousarray(np.concatenate([g["excluded"], g["special"]]), np.int32)
    fx4 = np.zeros((n, 4), np.float64)
    e_ex = hostlib.pmeh_exclusion(len(pairs), _ptr(pairs), _ptr(box), _ptr(pos4), _ptr(fx4), C.c_double(alpha), C.c_double(f_div))
    fx_ref, ex_ref = pme.ewald_exclusion(sd["coords"], g["charge"], box, pairs)
    assert np.abs(fx4[:, :3] - fx_ref).max() < 1e-9 * max(1.0, np.abs(fx_ref).max())
    assert abs(e_ex - ex_ref) < 1e-9 * abs(ex_ref)
    # end to end against OpenMM: pair terms from the C oracle, bonded from numpy, PME pieces from the device functions
    inters = [o.Inter(o.LJ, o.CUT_DISTANCE, 1.0, weight_special=float(g["lj14scale"]), use_neighbors=True),
              o.Inter(o.EWALD_REAL, o.CUT_DISTANCE, 1.0, weight_special=float(g["coulomb14scale"]), ewald_alpha=alpha,
                      use_neighbors=True)]
    f, e, _ = H.make_oracle(sd, inters, dtype=np.float64).forces_allpairs(sd["coords"])
    fb, eb = H.bonded_forces_oracle(g, sd["coords"])
    total = f + fb + f4[:, :3] + fx4[:, :3]
    assert np.linalg.norm(total[g["openmm_sample"]] - g["forces_all_pme_exact"], axis=1).max() < 1e-7
    e_tot = e + eb + e_recip + info["e_self"] + e_ex + o.lj_dispersion_correction_energy(g["sigma"], g["eps"], box, 1.0)
    assert abs(e_tot - float(g["energy_all_pme_exact"])) < 1e-5


def test_pme_device_functions_on_host_water3(hostlib):
    """Same chain on the reference's small PME case (orthorhombic 2.0 x 2.1 x 2.2 nm box, mesh 18 x 19 x 20): against
    the OpenMM literals of test/interactions.jl:1683-1697."""
    w = dict(np.load(os.path.join(ROOT, "tests", "golden", "water3.npz")))
    n = len(w["coords"])
    box = np.ascontiguousarray(w["box"], np.float64)
    rc = float(w["r_cut"])
    alpha = pme.pme_alpha(rc)
    K = np.array(pme.pme_mesh_dims(box, alpha), np.int32)
    bsm = [np.ascontiguousarray(m) for m in pme.bspline_moduli(5, tuple(K))]
    pos4 = np.ascontiguousarray(np.concatenate([w["coords"], w["charge"][:, None]], 1), np.float64)
    f_div = pme.COULOMB_CONST
    grid = np.zeros((K[0], K[1], K[2], 2), np.float64)
    hostlib.pmeh_spread(n, _ptr(K), _ptr(box), _ptr(pos4), _ptr(grid))
    S = np.fft.fftn(grid[..., 0])
    cg = np.ascontiguousarray(np.stack([S.real, S.imag], -1))
    e_recip = hostlib.pmeh_conv(_ptr(K), _ptr(box), C.c_double(f_div), C.c_double(alpha), _ptr(bsm[0]), _ptr(bsm[1]), _ptr(bsm[2]), _ptr(cg))
    pot = np.fft.ifftn(cg[..., 0] + 1j * cg[..., 1]) * K.prod()
    pg = np.ascontiguousarray(np.stack([pot.real, pot.imag], -1))
    f4 = np.zeros((n, 4), np.float64)
    hostlib.pmeh_interp(n, _ptr(K), _ptr(box), _ptr(pos4), _ptr(pg), _ptr(f4))
    pairs = np.ascontiguousarray(w["excluded"], np.int32)
    e_ex = hostlib.pmeh_exclusion(len(pairs), _ptr(pairs), _ptr(box), _ptr(pos4), _ptr(f4), C.c_double(alpha), C.c_double(f_div))
    s = o.OracleSystem(box=box, mass=w["mass"], charge=w["charge"], sigma=w["sigma"], eps=w["eps"],
                       inters=[o.Inter(o.EWALD_REAL, o.CUT_DISTANCE, rc, ewald_alpha=alpha, use_neighbors=True)],
                       excluded_pairs=w["excluded"], special_pairs=w["special"])
    f, e, _ = s.forces_allpairs(w["coords"])
    q = w["charge"]
    e_self = -f_div * (q ** 2).sum() * alpha / np.sqrt(np.pi) - f_div * np.pi * q.sum() ** 2 / (2 * box.prod() * alpha ** 2)
    assert np.linalg.norm(f + f4[:, :3] - w["forces_pme"], axis=1).max() < 1e-7
    assert abs(e + e_recip + e_self + e_ex - float(w["energy_pme"])) < 1e-8
