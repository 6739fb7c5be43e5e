// specific.cuh — host side of the terms added after the pair kernel, apart from PME (pme_host.cuh):
// BondedHost<T> holds the specific interaction lists (bonded.cuh) and launches their kernel; Dispersion holds the
// LJDispersionCorrection constants.
#pragma once
#include <algorithm>
#include <cmath>
#include <map>

#include "bonded.cuh"
#include "host_util.h"

namespace mb {

// specific (bonded) interaction lists: kind 0 bond (k, r0), 1 angle (k, theta0), 2 torsion (periodicity, phase, k)
template <typename T>
struct BondedHost {
    using T4 = typename VT<T>::T4;

    cudaStream_t stream_ = nullptr;  // the engine's stream
    int64_t n_[3] = {0, 0, 0};
    DevBuf d_idx_[3], d_par_[3], d_partial_, d_energy_;

    bool any() const { return n_[0] + n_[1] + n_[2] > 0; }
    double* energy() const { return d_energy_.as<double>(); }
    // mb_set_specific for a system of n_atoms atoms
    int set(int kind, int64_t n, const int32_t* idx, const double* par, int64_t n_atoms) {
        if (kind < 0 || kind > 2 || n < 0 || (n > 0 && (!idx || !par))) return set_error(MB_ERR_INVALID, "mb_set_specific: bad arguments");
        if (n_atoms <= 0) return set_error(MB_ERR_STATE, "mb_set_specific: set atoms first");
        const int na = kind + 2, np_ = (kind == 2) ? 3 : 2;
        std::vector<int> hidx((size_t)n * na);
        std::vector<T> hpar((size_t)n * np_);
        for (int64_t t = 0; t < n * na; t++) {
            int a = idx[t] - 1;  // 1-based in, like InteractionList{2,3,4}Atoms (src/types.jl:89-157)
            if (a < 0 || a >= n_atoms) return set_error(MB_ERR_INVALID, "mb_set_specific: atom index out of bounds");
            hidx[t] = a;
        }
        for (int64_t t = 0; t < n * np_; t++) hpar[t] = (T)par[t];
        n_[kind] = n;
        if (n > 0) {
            MB_CUDA(d_idx_[kind].ensure(hidx.size() * sizeof(int)));
            MB_CUDA(d_par_[kind].ensure(hpar.size() * sizeof(T)));
            MB_CUDA(cudaMemcpy(d_idx_[kind].p, hidx.data(), hidx.size() * sizeof(int), cudaMemcpyHostToDevice));
            MB_CUDA(cudaMemcpy(d_par_[kind].p, hpar.data(), hpar.size() * sizeof(T), cudaMemcpyHostToDevice));
        }
        int64_t mx = std::max(n_[0], std::max(n_[1], n_[2]));
        MB_CUDA(d_partial_.ensure((size_t)(3 * ((mx + BONDED_THREADS - 1) / BONDED_THREADS) + 8) * sizeof(double)));
        return MB_OK;
    }
    // add the bonded forces to f4 (slot_of: original -> slot index, or null in original order); with energy, the
    // per-kernel partials are summed into energy() (double, device), which starts from zero
    int launch(bool energy, const int* slot_of, const T4* pos4, T4* f4, const double box[3], int64_t& launches) {
        MB_CUDA(d_partial_.ensure(64 * sizeof(double)));  // (set sizes it for the lists; PME alone needs it to exist)
        BoxT bx;
        for (int d = 0; d < 3; d++) bx.L[d] = box[d];
        if (energy) {
            MB_CUDA(d_energy_.ensure(sizeof(double)));
            MB_CUDA(cudaMemsetAsync(d_energy_.p, 0, sizeof(double), stream_));
        }
        double* part = d_partial_.as<double>();
        BondedLists L;
        int total_blk = 0;
        for (int kind = 0; kind < 3; kind++) {
            L.n[kind] = (int)n_[kind];
            L.nblk[kind] = (L.n[kind] + BONDED_THREADS - 1) / BONDED_THREADS;
            L.idx[kind] = d_idx_[kind].as<int>();
            L.par[kind] = d_par_[kind].p;
            total_blk += L.nblk[kind];
        }
        if (total_blk > 0) {
            dispatch(energy, [&](auto EN) {
                bonded_kernel<T, EN><<<total_blk, BONDED_THREADS, 0, stream_>>>(L, slot_of, pos4, f4, bx, part);
                return MB_OK;
            });
            launches++;
            if (energy) {
                sum_partials_kernel<<<1, 256, 0, stream_>>>(total_blk, part, d_energy_.as<double>());
                launches++;
            }
        }
        MB_CUDA(cudaGetLastError());
        return MB_OK;
    }
};

// LJDispersionCorrection (general interaction; lennard_jones.jl:163-275)
struct Dispersion {
    double rc_ = 0, f6_ = 0, f12_ = 0;  // rc_ = 0: off
    bool ready_ = false;

    int set(double r_cut) {
        if (r_cut < 0) return set_error(MB_ERR_INVALID, "mb_set_lj_dispersion_correction: negative cutoff");
        rc_ = r_cut;
        ready_ = false;
        return MB_OK;
    }
    // factor_6 / factor_12 of the constructor (:170-226): means over all i <= j pairs, N (N + 1) / 2 terms, Lorentz sigma
    // and geometric epsilon without the zero shortcut; accumulated in double, grouped by distinct (sigma, eps)
    template <typename T>
    int prepare(int64_t n, const std::vector<T>& h_sigma, const std::vector<T>& h_eps_raw) {
        if (ready_ || rc_ <= 0) return MB_OK;
        if (n <= 0) return set_error(MB_ERR_STATE, "LJ dispersion correction: atoms not set");
        std::map<std::pair<double, double>, double> types;
        for (int64_t i = 0; i < n; i++) types[{(double)h_sigma[i], (double)h_eps_raw[i]}] += 1.0;
        std::vector<std::pair<std::pair<double, double>, double>> tv(types.begin(), types.end());
        double s6 = 0, s12 = 0;
        for (size_t a = 0; a < tv.size(); a++)
            for (size_t b = a; b < tv.size(); b++) {
                const double np = (a == b) ? tv[a].second * (tv[a].second + 1.0) / 2.0 : tv[a].second * tv[b].second;
                const double sig = (tv[a].first.first + tv[b].first.first) / 2.0;
                const double e = std::sqrt(tv[a].first.second * tv[b].first.second);
                const double sg6 = sig * sig * sig * sig * sig * sig;
                s6 += np * e * sg6;
                s12 += np * e * sg6 * sg6;
            }
        const double nd = (double)n, n_pairs = nd * (nd + 1.0) / 2.0, pi_ = 3.14159265358979323846;
        const double rc3 = rc_ * rc_ * rc_;
        f6_ = 8.0 * pi_ * nd * nd * (-(s6 / n_pairs) / (3.0 * rc3));
        f12_ = 8.0 * pi_ * nd * nd * ((s12 / n_pairs) / (9.0 * rc3 * rc3 * rc3));
        ready_ = true;
        return MB_OK;
    }
};

}  // namespace mb
