// pme_host.cuh — host side of PME (pme.cuh): the mesh / Ewald-parameter plan and PmeHost<T>, which owns the PME
// parameters, the cuFFT plan and the grid buffers of an engine and enqueues spread -> FFT -> convolution -> inverse FFT
// -> interpolation -> Ewald exclusions on the engine's stream.
#pragma once
#include <algorithm>
#include <cmath>

#include "bonded.cuh"
#include "dynlib.h"
#include "host_util.h"
#include "pme.cuh"

namespace mb {

// ---------------------------------------------------------------------------------------------
// PME plan (pure host logic, exported as mb_pme_plan so it is tested on the CPU against oracle/pme.py):
// alpha = sqrt(-ln(2 tol)) / rc (ewald.jl:373), mesh dims = max(6, ceil(2 alpha L / (3 tol^0.2))) (:484-487),
// B-spline moduli (:311-361).
// ---------------------------------------------------------------------------------------------
static void pme_plan_host(const double box[3], double r_cut, double error_tol, int order, double* alpha_out, int K[3],
                          std::vector<double> moduli[3]) {
    const double alpha = std::sqrt(-std::log(2.0 * error_tol)) / r_cut;
    *alpha_out = alpha;
    for (int d = 0; d < 3; d++) K[d] = std::max((int)std::ceil(2.0 * alpha * box[d] / (3.0 * std::pow(error_tol, 0.2))), 6);
    std::vector<double> data(order, 0.0);
    data[0] = 1.0;
    for (int k = 3; k <= order; k++) {
        const double d = 1.0 / (k - 1.0);
        data[k - 1] = 0.0;
        for (int l = 1; l <= k - 2; l++) data[k - l - 1] = d * (l * data[k - l - 2] + (k - l) * data[k - l - 1]);
        data[0] *= d;
    }
    const double two_pi = 6.283185307179586476925;
    for (int d = 0; d < 3; d++) {
        const int nd = K[d];
        std::vector<double> bs((size_t)std::max(nd, order + 1), 0.0);
        std::vector<double>& mod = moduli[d];
        mod.assign(nd, 0.0);
        for (int i = 0; i < order; i++) bs[i + 1] = data[i];
        for (int i = 0; i < nd; i++) {
            double sc = 0, ss = 0;
            for (int j = 0; j < nd; j++) {
                const double arg = two_pi * i * j / nd;
                sc += bs[j] * std::cos(arg);
                ss += bs[j] * std::sin(arg);
            }
            mod[i] = sc * sc + ss * ss;
        }
        for (int i = 0; i < nd; i++)
            if (mod[i] < 1e-7) mod[i] = 0.5 * (mod[(i - 1 + nd) % nd] + mod[(i + 1) % nd]);
    }
}

// PME reciprocal space + Ewald exclusions (pme.cuh; SURVEY.md §8(f)-3)
template <typename T>
struct PmeHost {
    using T4 = typename VT<T>::T4;
    using T2 = typename VT<T>::T2;

    cudaStream_t stream_ = nullptr;  // the engine's stream
    bool on_ = false, ready_ = false;
    double rc_ = 0, tol_ = 0, epsr_ = 1, alpha_ = 0, self_e_ = 0, ke_ = 138.93545764;
    PmeGeom g_ = {{0, 0, 0}, {0, 0, 0}};
    int plan_ = -1;
    std::vector<int> pairs_;
    DevBuf d_grid_, d_bsm_[3], d_partial_, d_pairs_;

    void destroy_plan() {
        if (plan_ >= 0 && g_cufft.Destroy) g_cufft.Destroy(plan_);
    }
    // mb_set_pme for a system of n atoms; order 0 switches PME off
    int set(double r_cut, double error_tol, int order, double eps_r, int64_t n_pairs, const int32_t* pi, const int32_t* pj, int64_t n) {
        if (order == 0) { on_ = false; return MB_OK; }
        if (order != PME_ORDER) return set_error(MB_ERR_INVALID, "mb_set_pme: only B-spline order 5 is implemented (the reference's default)");
        if (!(r_cut > 0) || !(error_tol > 0 && error_tol < 0.5) || !(eps_r > 0) || n_pairs < 0 || (n_pairs > 0 && (!pi || !pj)))
            return set_error(MB_ERR_INVALID, "mb_set_pme: bad arguments");
        if (n <= 0) return set_error(MB_ERR_STATE, "mb_set_pme: set atoms first");
        if (!g_cufft.load()) return set_error(MB_ERR_INVALID, "mb_set_pme: libcufft could not be loaded");
        pairs_.resize((size_t)2 * n_pairs);
        for (int64_t k = 0; k < n_pairs; k++) {
            const int a = pi[k] - 1, b = pj[k] - 1;  // 1-based in
            if (a < 0 || b < 0 || a >= n || b >= n) return set_error(MB_ERR_INVALID, "mb_set_pme: pair index out of bounds");
            pairs_[2 * k] = a;
            pairs_[2 * k + 1] = b;
        }
        rc_ = r_cut; tol_ = error_tol; epsr_ = eps_r;
        on_ = true;
        ready_ = false;
        return MB_OK;
    }
    // grid dimensions, B-spline moduli, plan, self energy: ewald.jl:363-421 (constructor) and :947-956
    int prepare(const double box[3], const std::vector<T>& h_charge) {
        bool same_box = ready_;
        for (int d = 0; d < 3; d++) same_box = same_box && (g_.L[d] == box[d]);
        if (same_box) return MB_OK;
        std::vector<double> moduli[3];
        pme_plan_host(box, rc_, tol_, PME_ORDER, &alpha_, g_.K, moduli);
        for (int d = 0; d < 3; d++) {
            g_.L[d] = box[d];
            MB_CUDA(d_bsm_[d].ensure(moduli[d].size() * sizeof(double)));
            MB_CUDA(cudaMemcpy(d_bsm_[d].p, moduli[d].data(), moduli[d].size() * sizeof(double), cudaMemcpyHostToDevice));
        }
        const size_t total = (size_t)g_.K[0] * g_.K[1] * g_.K[2];
        MB_CUDA(d_grid_.ensure(total * sizeof(T2)));
        const int conv_blk = (int)((total + PME_THREADS - 1) / PME_THREADS);
        const int ex_blk = (int)((pairs_.size() / 2 + PME_THREADS - 1) / PME_THREADS);
        MB_CUDA(d_partial_.ensure((size_t)(conv_blk + ex_blk + 8) * sizeof(double)));
        if (!pairs_.empty()) {
            MB_CUDA(d_pairs_.ensure(pairs_.size() * sizeof(int)));
            MB_CUDA(cudaMemcpy(d_pairs_.p, pairs_.data(), pairs_.size() * sizeof(int), cudaMemcpyHostToDevice));
        }
        if (plan_ >= 0) { g_cufft.Destroy(plan_); plan_ = -1; }
        const int type = (sizeof(T) == 4) ? 0x29 /* CUFFT_C2C */ : 0x69 /* CUFFT_Z2Z */;
        if (g_cufft.Plan3d(&plan_, g_.K[0], g_.K[1], g_.K[2], type) != 0) {
            plan_ = -1;
            return set_error(MB_ERR_CUDA, "cufftPlan3d failed");
        }
        if (g_cufft.SetStream(plan_, stream_) != 0) return set_error(MB_ERR_CUDA, "cufftSetStream failed");
        // self and neutralising-background energy (ewald.jl:947-956)
        double qs = 0, q2 = 0;
        for (size_t i = 0; i < h_charge.size(); i++) { qs += (double)h_charge[i]; q2 += (double)h_charge[i] * (double)h_charge[i]; }
        const double f_div = ke_ / epsr_;
        const double V = box[0] * box[1] * box[2];
        const double pi_ = 3.14159265358979323846;
        self_e_ = -f_div * q2 * alpha_ / std::sqrt(pi_) - f_div * pi_ * qs * qs / (2.0 * V * alpha_ * alpha_);
        ready_ = true;
        return MB_OK;
    }
    // add the reciprocal-space and exclusion forces of the n atoms in pos4 to f4 (slot_of: original -> slot index, or
    // null in original order); with energy, add the PME energy to *energy_acc (device double)
    int launch(bool energy, int64_t n, const double box[3], const std::vector<T>& h_charge, const T4* pos4, T4* f4,
               const int* slot_of, double* energy_acc, int64_t& launches) {
        MB_TRY(prepare(box, h_charge));
        const int nb = (int)((n + PME_THREADS - 1) / PME_THREADS);
        const size_t total = (size_t)g_.K[0] * g_.K[1] * g_.K[2];
        const int conv_blk = (int)((total + PME_THREADS - 1) / PME_THREADS);
        const int n_ex = (int)(pairs_.size() / 2);
        const int ex_blk = (n_ex + PME_THREADS - 1) / PME_THREADS;
        const double f_div = ke_ / epsr_;
        const double pi_ = 3.14159265358979323846;
        const double factor = pi_ * pi_ / (alpha_ * alpha_);
        const double boxfactor = pi_ * box[0] * box[1] * box[2];
        double* part = d_partial_.as<double>();
        T2* grid = d_grid_.as<T2>();
        MB_CUDA(cudaMemsetAsync(grid, 0, total * sizeof(T2), stream_));
        pme_spread_kernel<T><<<nb, PME_THREADS, 0, stream_>>>((int)n, g_, pos4, grid);
        auto fft = [&](int dir) -> int {
            const int rc = (sizeof(T) == 4) ? g_cufft.ExecC2C(plan_, grid, grid, dir) : g_cufft.ExecZ2Z(plan_, grid, grid, dir);
            return rc == 0 ? MB_OK : set_error(MB_ERR_CUDA, "cufftExec failed");
        };
        MB_TRY(fft(-1));
        dispatch(energy, [&](auto EN) {
            pme_conv_kernel<T, EN><<<conv_blk, PME_THREADS, 0, stream_>>>(g_, f_div, factor, boxfactor, d_bsm_[0].as<double>(),
                                                                          d_bsm_[1].as<double>(), d_bsm_[2].as<double>(), grid, part);
            return MB_OK;
        });
        MB_TRY(fft(1));
        pme_interp_kernel<T><<<nb, PME_THREADS, 0, stream_>>>((int)n, g_, pos4, grid, f4);
        launches += 3;
        if (n_ex > 0) {
            dispatch(energy, [&](auto EN) {
                ewald_exclusion_kernel<T, EN><<<ex_blk, PME_THREADS, 0, stream_>>>(n_ex, d_pairs_.as<int>(), slot_of, pos4, f4, g_,
                                                                                   alpha_, f_div, part + conv_blk);
                return MB_OK;
            });
            launches++;
        }
        if (energy) {
            sum_partials_kernel<<<1, 256, 0, stream_>>>(conv_blk + (n_ex > 0 ? ex_blk : 0), part, energy_acc);
            add_const_kernel<<<1, 1, 0, stream_>>>(energy_acc, self_e_);
            launches += 2;
        }
        MB_CUDA(cudaGetLastError());
        return MB_OK;
    }
};

}  // namespace mb
