// engine.cu — host side of libmollyb200: Engine<T> (parameter digestion, geometry and capacity choice, the rebuild
// pipeline driver, force dispatch, the MD step and its CUDA graph, the small reductions) and the C ABI declared in
// include/mollyb200.h. The other host units are headers included into this one translation unit: host_util.h (errors,
// status macros, device buffers, timing, the runtime -> template dispatch), dynlib.h (NCCL and cuFFT bound with
// dlopen), decomp.cuh (slab plan and Decomp<T>, all multi-GPU state and transport), pme_host.cuh (PME plan and
// PmeHost<T>) and specific.cuh (bonded lists and the LJ dispersion correction). Kernels live in force.cuh, cells.cuh,
// vv.cuh, bonded.cuh, pme.cuh and peer.cuh.
//
// There is deliberately no CPU code path: every entry point needs a CUDA device.
#include <algorithm>
#include <climits>
#include <memory>

#include "cells.cuh"
#include "common.cuh"
#include "decomp.cuh"
#include "dynlib.h"
#include "force.cuh"
#include "host_util.h"
#include "pair.cuh"
#include "pme_host.cuh"
#include "specific.cuh"
#include "vv.cuh"

namespace mb {

// Kernel variants, as lists for dispatch(). The brick force kernel additionally has UNIFORM = true for COUL_NONE only.
// Experiment builds (-DMB_EXP_FAST, profiles/r02_experiments.md) instantiate only the LJ and LJ + CRF brick kernels with
// plain cutoffs, and only in f32 (mb_ctx_create).
using AllCoulKinds = Vals<COUL_NONE, COUL_PLAIN, COUL_CRF, COUL_EWALD>;
using AllCutModes = Vals<CUTM_PLAIN, CUTM_SHIFTED, CUTM_TWO_POINT>;
#ifdef MB_EXP_FAST
using BrickCoulKinds = Vals<COUL_NONE, COUL_CRF>;
using BrickCutModes = Vals<CUTM_PLAIN>;
#else
using BrickCoulKinds = AllCoulKinds;
using BrickCutModes = AllCutModes;
#endif

// Environment switches (diagnostics and tuning aids, INTEGRATION.md), read once when a context is created.
static bool env_starts(const char* name, char c) {
    const char* e = getenv(name);
    return e && e[0] == c;
}
struct EnvSwitches {
    bool graph = !env_starts("MOLLYB200_NO_GRAPH", '1');             // else the plain-stream MD step
    bool static_sched = env_starts("MOLLYB200_STATIC_SCHED", '1');   // force kernel takes bricks round-robin, not by ticket
    bool p2p = !env_starts("MOLLYB200_P2P", '0');                    // else the NCCL transport for decomposed runs
    int max_nbuf = getenv("MOLLYB200_NBUF") ? atoi(getenv("MOLLYB200_NBUF")) : INT_MAX;  // cap on the force kernel's ring
};

class EngineBase {
   public:
    virtual ~EngineBase() {}
    virtual int set_atoms_aos(int64_t n, const void* aos) = 0;
    virtual int set_atoms_soa(int64_t n, const void* mass, const void* charge, const void* sigma, const void* eps) = 0;
    virtual int set_box(const double side[3]) = 0;
    virtual int set_box_triclinic(const double basis[9]) = 0;
    virtual int set_inters(int n, const mb_inter_t* in) = 0;
    virtual int set_exceptions(int64_t ne, const int32_t* ei, const int32_t* ej, int64_t ns, const int32_t* si,
                               const int32_t* sj) = 0;
    virtual int set_neighbor_policy(double r_list, int rebuild_every) = 0;
    virtual int forces_energy(const void* coords, void* fs, void* pe, void* vir, int64_t step_n, bool with_specific) = 0;
    virtual int simulate_vv(void* coords, void* vels, const mb_vv_params_t* p) = 0;
    virtual int remove_cm(void* vels) = 0;
    virtual int kinetic_energy(const void* vels, double* out) = 0;
    virtual int rebuild(const void* coords) = 0;
    virtual int stats(mb_stats_t* out) = 0;
    virtual int synchronize() = 0;
    virtual int set_capacity_scale(double s) = 0;
    virtual int set_launch_config(const int32_t bd[3], int32_t lpa) = 0;
    virtual int set_profiling(int enable) = 0;
    virtual int comm_init(const void* uid, int rank, int nranks) = 0;
    virtual int set_specific(int kind, int64_t n, const int32_t* idx, const double* par) = 0;
    virtual int set_pme(double r_cut, double error_tol, int order, double eps_r, int64_t n_pairs, const int32_t* pi, const int32_t* pj) = 0;
    virtual int set_dispersion(double r_cut) = 0;
    virtual int random_velocities(void* vels, double kT, uint64_t ctr1, uint64_t key) = 0;
    virtual int kinetic_tensor(const void* vels, double* out9) = 0;
};

template <typename T>
class Engine : public EngineBase {
    using T4 = typename VT<T>::T4;
    using T2 = typename VT<T>::T2;

   public:
    Engine(int device, cudaStream_t stream) : stream_(stream) {
        cudaDeviceProp prop;
        cudaGetDeviceProperties(&prop, device);
        sm_count_ = prop.multiProcessorCount;
        smem_optin_ = prop.sharedMemPerBlockOptin;
        for (int d = 0; d < 3; d++) box_[d] = 0;
        if (!stream_) {
            // a real (blocking) stream: graph capture is not allowed on the legacy default stream, and a blocking
            // stream keeps the implicit ordering with work the caller issues on the default stream
            if (cudaStreamCreateWithFlags(&stream_, cudaStreamDefault) == cudaSuccess) own_stream_ = true;
            else stream_ = nullptr;
        }
        prof_.stream = dc_.stream_ = pme_.stream_ = bonded_.stream_ = stream_;
    }
    ~Engine() override {
        destroy_graph();
        dc_.p2p_close();
        pme_.destroy_plan();
        if (own_stream_) cudaStreamDestroy(stream_);
    }

    // ------------------------------------------------------------------------------------------
    int set_atoms_aos(int64_t n, const void* aos) override {
        if (n <= 0 || !aos) return set_error(MB_ERR_INVALID, "mb_set_atoms: n <= 0 or null atoms");
        // Atom{Int32,T,T,T,T,T}: int32 index, int32 atom_type, T mass, T charge, T sigma, T eps, T lambda, int32 role
        const size_t rec = (sizeof(T) == 4) ? 32 : 56;
        std::vector<unsigned char> host((size_t)n * rec);
        MB_CUDA(cudaMemcpy(host.data(), aos, host.size(), cudaMemcpyDefault));
        h_mass_.resize(n); h_charge_.resize(n); h_sigma_.resize(n); h_eps_.resize(n); h_eps_raw_.resize(n);
        for (int64_t i = 0; i < n; i++) {
            const unsigned char* r = host.data() + (size_t)i * rec;
            T vals[5];
            memcpy(vals, r + 8, 5 * sizeof(T));
            h_mass_[i] = vals[0];
            h_charge_[i] = vals[1];
            h_sigma_[i] = vals[2];
            h_eps_[i] = (vals[4] == (T)0) ? (T)0 : vals[3];  // lambda == 0 -> LJ zero shortcut (mixing.jl:7-11)
            h_eps_raw_[i] = vals[3];
        }
        n_ = n;
        dirty_ = true;
        return MB_OK;
    }
    int set_atoms_soa(int64_t n, const void* mass, const void* charge, const void* sigma, const void* eps) override {
        if (n <= 0 || !mass || !charge || !sigma || !eps)
            return set_error(MB_ERR_INVALID, "mb_set_atoms_soa: n <= 0 or null array");
        h_mass_.resize(n); h_charge_.resize(n); h_sigma_.resize(n); h_eps_.resize(n);
        MB_CUDA(cudaMemcpy(h_mass_.data(), mass, n * sizeof(T), cudaMemcpyDefault));
        MB_CUDA(cudaMemcpy(h_charge_.data(), charge, n * sizeof(T), cudaMemcpyDefault));
        MB_CUDA(cudaMemcpy(h_sigma_.data(), sigma, n * sizeof(T), cudaMemcpyDefault));
        MB_CUDA(cudaMemcpy(h_eps_.data(), eps, n * sizeof(T), cudaMemcpyDefault));
        h_eps_raw_ = h_eps_;
        n_ = n;
        dirty_ = true;
        return MB_OK;
    }
    int set_box(const double side[3]) override {
        for (int d = 0; d < 3; d++) {
            if (!(side[d] > 0) || std::isinf(side[d]))
                return set_error(MB_ERR_INVALID, "mb_set_box: side lengths must be finite and > 0 (CubicBoundary)");
            box_[d] = side[d];
        }
        memset(&tric_, 0, sizeof(tric_));
        dirty_ = true;
        return MB_OK;
    }
    // TriclinicBoundary(bv1, bv2, bv3) (src/spatial.jl:165-215): lower-triangular basis, positive diagonal. Such systems run
    // on the no-list kernel (minimum image :528-534, wrap :584-600); the cell-list path is for Cubic/Rectangular boxes.
    int set_box_triclinic(const double b[9]) override {
        if (!(b[0] > 0) || b[1] != 0 || b[2] != 0)
            return set_error(MB_ERR_INVALID, "mb_set_box_triclinic: first basis vector must be along the x-axis with a positive x component");
        if (!(b[4] > 0) || b[5] != 0)
            return set_error(MB_ERR_INVALID, "mb_set_box_triclinic: second basis vector must be in the xy plane with a positive y component");
        if (!(b[8] > 0)) return set_error(MB_ERR_INVALID, "mb_set_box_triclinic: third basis vector must have a positive z component");
        for (int k = 0; k < 9; k++)
            if (std::isinf(b[k]) || std::isnan(b[k])) return set_error(MB_ERR_INVALID, "mb_set_box_triclinic: infinite boundaries are not supported");
        Tric<T> t;
        memset(&t, 0, sizeof(t));
        t.on = 1;
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) t.bv[i][j] = (T)b[3 * i + j];
        t.rs[0] = (T)(1.0 / b[0]); t.rs[1] = (T)(1.0 / b[4]); t.rs[2] = (T)(1.0 / b[8]);
        const double by = b[4], bz = b[5], cy = b[7], cz = b[8];
        t.cot_bprojyz_cprojyz = (T)std::fabs((by * cy + bz * cz) / (by * cz - bz * cy));
        t.cprojxy_x_over_z = (T)(b[6] / std::fabs(b[8]));
        t.cprojxy_y_over_z = (T)(b[7] / std::fabs(b[8]));
        t.cot_a_b = (T)(b[3] / b[4]);
        tric_ = t;
        box_[0] = b[0]; box_[1] = b[4]; box_[2] = b[8];  // heights: volume = their product
        dirty_ = true;
        return MB_OK;
    }
    int set_inters(int n, const mb_inter_t* in) override {
        if (n < 0 || (n > 0 && !in)) return set_error(MB_ERR_INVALID, "mb_set_inters: bad arguments");
        int n_lj = 0, n_c = 0;
        for (int k = 0; k < n; k++) {
            if (in[k].kind == MB_LJ) n_lj++;
            else if (in[k].kind == MB_COULOMB || in[k].kind == MB_CRF || in[k].kind == MB_EWALD_REAL) n_c++;
            else return set_error(MB_ERR_INVALID, "mb_set_inters: unknown interaction kind");
            if (in[k].cutoff_kind < MB_CUT_NONE || in[k].cutoff_kind > MB_CUT_POLYNOMIAL)
                return set_error(MB_ERR_INVALID, "mb_set_inters: unsupported cutoff kind");
            if (in[k].cutoff_kind >= MB_CUT_CUBIC_SPLINE) {
                // CubicSplineCutoff / PolynomialCutoff constructors, src/cutoffs.jl:181-187, :239-245
                if (in[k].kind != MB_LJ && in[k].kind != MB_COULOMB)
                    return set_error(MB_ERR_INVALID, "mb_set_inters: two-point cutoffs apply to LennardJones and Coulomb only");
                if (!(in[k].r_act > 0) || !(in[k].r_cut > in[k].r_act))
                    return set_error(MB_ERR_INVALID, "mb_set_inters: the cutoff radius must be larger than the activation radius");
            }
            if (in[k].kind == MB_LJ && in[k].eps_mix != MB_MIX_GEOMETRIC)
                return set_error(MB_ERR_INVALID, "mb_set_inters: only geometric epsilon mixing is supported");
        }
        if (n_lj > 1 || n_c > 1)
            return set_error(MB_ERR_INVALID, "mb_set_inters: at most one LJ and one Coulomb-family interaction");
        inters_.assign(in, in + n);
        dirty_ = true;
        return MB_OK;
    }
    int set_exceptions(int64_t ne, const int32_t* ei, const int32_t* ej, int64_t ns, const int32_t* si,
                       const int32_t* sj) override {
        if (n_ <= 0) return set_error(MB_ERR_STATE, "mb_set_exceptions: set atoms first");
        auto build = [&](int64_t m, const int32_t* a, const int32_t* b, std::vector<int>& ptr, std::vector<int>& idx,
                         const std::vector<int>* skip_ptr, const std::vector<int>* skip_idx) -> int {
            std::vector<std::pair<int, int>> pr;
            pr.reserve(2 * m);
            for (int64_t k = 0; k < m; k++) {
                int i = a[k] - 1, j = b[k] - 1;  // 1-based in, 0-based inside
                if (i < 0 || j < 0 || i >= n_ || j >= n_)
                    return set_error(MB_ERR_INVALID, "mb_set_exceptions: index out of bounds");
                if (i == j) continue;
                if (skip_ptr && !skip_ptr->empty()) {
                    bool ex = false;
                    for (int q = (*skip_ptr)[i]; q < (*skip_ptr)[i + 1]; q++) ex |= ((*skip_idx)[q] == j);
                    if (ex) continue;  // excluded wins over special
                }
                pr.emplace_back(i, j);
                pr.emplace_back(j, i);
            }
            std::sort(pr.begin(), pr.end());
            pr.erase(std::unique(pr.begin(), pr.end()), pr.end());
            ptr.assign(n_ + 1, 0);
            idx.resize(pr.size());
            for (auto& p : pr) ptr[p.first + 1]++;
            for (int64_t i = 0; i < n_; i++) ptr[i + 1] += ptr[i];
            for (size_t k = 0; k < pr.size(); k++) idx[k] = pr[k].second;
            return MB_OK;
        };
        MB_TRY(build(ne, ei, ej, ex_ptr_, ex_idx_, nullptr, nullptr));
        MB_TRY(build(ns, si, sj, sp_ptr_, sp_idx_, &ex_ptr_, &ex_idx_));
        if (ex_idx_.empty()) ex_ptr_.clear();
        if (sp_idx_.empty()) sp_ptr_.clear();
        dirty_ = true;
        return MB_OK;
    }
    int set_neighbor_policy(double r_list, int rebuild_every) override {
        if (r_list < 0 || rebuild_every < 0) return set_error(MB_ERR_INVALID, "mb_set_neighbor_policy: negative value");
        r_list_ = r_list;
        rebuild_every_ = rebuild_every;
        dirty_ = true;
        return MB_OK;
    }
    int set_capacity_scale(double s) override {
        if (!(s >= 1.0)) return set_error(MB_ERR_INVALID, "capacity scale must be >= 1");
        cap_scale_ = s;
        have_list_ = false;
        return MB_OK;
    }
    int set_launch_config(const int32_t bd[3], int32_t lpa) override {
        for (int d = 0; d < 3; d++) {
            if (bd[d] < 0 || bd[d] > 8) return set_error(MB_ERR_INVALID, "brick dims must be in 0..8");
            user_b_[d] = bd[d];
        }
        if (!(lpa == 0 || lpa == 8))
            return set_error(MB_ERR_INVALID, "lanes_per_atom must be 0 (default) or 8: the 4- and 16-lane variants were measured slower and removed");
        have_list_ = false;
        dirty_ = true;
        return MB_OK;
    }
    int set_profiling(int enable) override {
        prof_.reset();
        prof_.enabled = enable != 0;
        return MB_OK;
    }
    int synchronize() override {
        MB_CUDA(cudaStreamSynchronize(stream_));
        return MB_OK;
    }

    // ------------------------------------------------------------------------------------------
    // digest parameters -> kernel constants, allocate per-atom state
    int prepare() {
        if (!dirty_) return MB_OK;
        if (n_ <= 0) return set_error(MB_ERR_STATE, "atoms not set");
        if (!(box_[0] > 0)) return set_error(MB_ERR_STATE, "box not set");
        if (n_ > 2000000000LL) return set_error(MB_ERR_INVALID, "too many atoms");
        memset(&P_, 0, sizeof(P_));
        const double inf = std::numeric_limits<double>::infinity();
        bool all_nl = !inters_.empty();
        double max_rc = 0;
        bool any_nocut_nl = false;
        for (auto& in : inters_) {
            if (!in.use_neighbors) all_nl = false;
            if (in.cutoff_kind != MB_CUT_NONE || in.kind == MB_CRF || in.kind == MB_EWALD_REAL)
                max_rc = std::max(max_rc, in.r_cut);
            else if (in.use_neighbors)
                any_nocut_nl = true;
        }
        const double min_box = std::min(box_[0], std::min(box_[1], box_[2]));
        path_ = (all_nl && r_list_ > 0 && min_box >= 2.5 * r_list_ && n_ >= 64 && !tric_.on) ? 1 : 0;
        if (tric_.on && has_specific())
            return set_error(MB_ERR_INVALID, "TriclinicBoundary: specific interaction lists and PME are not supported by this engine");
        if (tric_.on && dc_.decomposed()) return set_error(MB_ERR_INVALID, "TriclinicBoundary: not available in decomposed (multi-GPU) runs");
        if (path_ == 1 && max_rc > r_list_)
            return set_error(MB_ERR_INVALID, "neighbour list radius is smaller than an interaction cutoff");
        skin_ = (path_ == 1) ? (any_nocut_nl ? 0.0 : r_list_ - max_rc) : 0.0;
        P_.has_lj = 0;
        P_.coul_kind = COUL_NONE;
        P_.lj_rc2 = (T)0;
        P_.c_rc2 = (T)0;
        cutm_ = CUTM_PLAIN;
        bool geo_sigma = false;
        for (auto& in : inters_) {
            // effective cutoff: NoCutoff with a neighbour list -> the finder radius (ext/MollyCUDAExt.jl:1691)
            double rc = inf;
            int ck = in.cutoff_kind;
            if (in.kind == MB_CRF || in.kind == MB_EWALD_REAL) {
                rc = in.r_cut;
                ck = MB_CUT_DISTANCE;
            } else if (ck != MB_CUT_NONE) {
                rc = in.r_cut;
            } else if (in.use_neighbors && r_list_ > 0) {
                rc = r_list_;
            }
            if (ck >= MB_CUT_CUBIC_SPLINE) cutm_ = CUTM_TWO_POINT;
            else if (ck >= MB_CUT_SHIFTED_POTENTIAL && cutm_ == CUTM_PLAIN) cutm_ = CUTM_SHIFTED;
            if (in.kind == MB_LJ) {
                P_.has_lj = 1;
                P_.lj_cut_kind = ck;
                P_.lj_rc = (T)rc; P_.lj_rc2 = (T)(rc * rc); P_.lj_inv_rc = (T)(1.0 / rc); P_.lj_inv_rc2 = (T)(1.0 / (rc * rc));
                P_.lj_ra = (T)in.r_act; P_.lj_inv_ra2 = (in.r_act > 0) ? (T)(1.0 / (in.r_act * in.r_act)) : (T)0;
                P_.lj_w14 = (T)in.weight_special;
                P_.lj_nl = in.use_neighbors ? 1 : 0;
                geo_sigma = (in.sigma_mix == MB_MIX_GEOMETRIC);
            } else {
                P_.coul_kind = (in.kind == MB_COULOMB) ? COUL_PLAIN : (in.kind == MB_CRF ? COUL_CRF : COUL_EWALD);
                P_.coul_cut_kind = ck;
                P_.c_rc = (T)rc; P_.c_rc2 = (T)(rc * rc); P_.c_inv_rc = (T)(1.0 / rc); P_.c_inv_rc2 = (T)(1.0 / (rc * rc));
                P_.ke = (T)in.coulomb_const;
                P_.c_w14 = (T)in.weight_special;
                P_.c_nl = in.use_neighbors ? 1 : 0;
                P_.alpha = (T)in.ewald_alpha;
                P_.c_ra = (T)in.r_act;
                P_.approx_erfc = (in.kind == MB_EWALD_REAL && in.approx_erfc) ? 1 : 0;
                if (in.kind == MB_CRF) {
                    double e = in.solvent_dielectric;
                    double krf, crf;
                    if (std::isinf(e)) { krf = 1.0 / (2.0 * rc * rc * rc); crf = 3.0 / (2.0 * rc); }
                    else { krf = (1.0 / (rc * rc * rc)) * (e - 1.0) / (2.0 * e + 1.0); crf = (1.0 / rc) * (3.0 * e) / (2.0 * e + 1.0); }
                    P_.krf = (T)krf;
                    P_.crf = (T)crf;
                }
            }
        }
        P_.geo_sigma = geo_sigma ? 1 : 0;
        // per-atom LJ parts (zero shortcut folded into a zero eps part)
        std::vector<T2> ljp(n_);
        bool uniform = true;
        for (int64_t i = 0; i < n_; i++) {
            T s = h_sigma_[i], e = h_eps_[i];
            bool zero = (!P_.has_lj) || s == (T)0 || e == (T)0;
            ljp[i].x = zero ? (T)0 : (geo_sigma ? (T)std::sqrt((double)s) : s / (T)2);
            ljp[i].y = zero ? (T)0 : (T)std::sqrt((double)e);
            if (h_sigma_[i] != h_sigma_[0] || h_eps_[i] != h_eps_[0]) uniform = false;
        }
        if (!P_.has_lj || h_sigma_[0] == (T)0 || h_eps_[0] == (T)0) uniform = uniform && !P_.has_lj;
        P_.uniform_lj = (uniform && P_.coul_kind == COUL_NONE) ? 1 : 0;
        if (P_.uniform_lj) {
            P_.uni_sig2 = P_.has_lj ? h_sigma_[0] * h_sigma_[0] : (T)0;
            P_.uni_eps = P_.has_lj ? h_eps_[0] : (T)0;
            const double s6 = std::pow((double)h_sigma_[0], 6.0), e0 = P_.has_lj ? (double)h_eps_[0] : 0.0;
            P_.uni_A = (T)(48.0 * e0 * s6 * s6);
            P_.uni_B = (T)(24.0 * e0 * s6);
        }
        total_mass_ = 0;
        for (int64_t i = 0; i < n_; i++) total_mass_ += (double)h_mass_[i];

        // per-atom device arrays (original order)
        const size_t np = (size_t)n_ + 16;
        MB_CUDA(d_mass_in_.ensure(np * sizeof(T)));
        MB_CUDA(d_charge_in_.ensure(np * sizeof(T)));
        MB_CUDA(d_ljp_in_.ensure(np * sizeof(T2)));
        MB_CUDA(cudaMemcpyAsync(d_mass_in_.p, h_mass_.data(), n_ * sizeof(T), cudaMemcpyHostToDevice, stream_));
        MB_CUDA(cudaMemcpyAsync(d_charge_in_.p, h_charge_.data(), n_ * sizeof(T), cudaMemcpyHostToDevice, stream_));
        MB_CUDA(cudaMemcpyAsync(d_ljp_in_.p, ljp.data(), n_ * sizeof(T2), cudaMemcpyHostToDevice, stream_));
        MB_CUDA(cudaStreamSynchronize(stream_));  // ljp is a local
        // slot-order state
        MB_CUDA(d_pos4_.ensure(np * sizeof(T4)));
        MB_CUDA(d_vel4_.ensure(np * sizeof(T4)));
        MB_CUDA(d_f4_.ensure(np * sizeof(T4)));
        MB_CUDA(d_xref4_.ensure(np * sizeof(T4)));
        MB_CUDA(d_lj2_.ensure(np * sizeof(T2)));
        MB_CUDA(d_orig_.ensure(np * sizeof(int)));
        MB_CUDA(d_inv_orig_.ensure(np * sizeof(int)));
        MB_CUDA(d_mass_.ensure(np * sizeof(T)));
        MB_CUDA(cudaMemsetAsync(d_f4_.p, 0, np * sizeof(T4), stream_));
        MB_CUDA(cudaMemsetAsync(d_lj2_.p, 0, np * sizeof(T2), stream_));
        MB_CUDA(cudaMemsetAsync(d_pos4_.p, 0, np * sizeof(T4), stream_));
        MB_CUDA(d_ctl_.ensure(sizeof(Control)));
        MB_CUDA(cudaMemsetAsync(d_ctl_.p, 0, sizeof(Control), stream_));
        MB_CUDA(d_cm_.ensure(sizeof(CmState<T>)));
        MB_CUDA(cudaMemsetAsync(d_cm_.p, 0, sizeof(CmState<T>), stream_));
        MB_CUDA(d_stage_a_.ensure(3 * np * sizeof(T)));
        MB_CUDA(d_stage_b_.ensure(3 * np * sizeof(T)));
        MB_CUDA(d_stage_c_.ensure(3 * np * sizeof(T)));
        // exclusion CSR
        auto up = [&](DevBuf& b, const std::vector<int>& v) -> cudaError_t {
            if (v.empty()) return cudaSuccess;
            cudaError_t e = b.ensure(v.size() * sizeof(int));
            if (e != cudaSuccess) return e;
            return cudaMemcpy(b.p, v.data(), v.size() * sizeof(int), cudaMemcpyHostToDevice);
        };
        MB_CUDA(up(d_ex_ptr_, ex_ptr_)); MB_CUDA(up(d_ex_idx_, ex_idx_));
        MB_CUDA(up(d_sp_ptr_, sp_ptr_)); MB_CUDA(up(d_sp_idx_, sp_idx_));
        max_special_host_ = 0;
        for (size_t i = 0; i + 1 < sp_ptr_.size(); i++) max_special_host_ = std::max(max_special_host_, sp_ptr_[i + 1] - sp_ptr_[i]);
        const int vvb = (int)((n_ + VV_THREADS - 1) / VV_THREADS);
        MB_CUDA(d_partial_.ensure((size_t)std::max(vvb, 2048) * 8 * sizeof(double)));
        have_list_ = false;
        dirty_ = false;
        return MB_OK;
    }

    const int* ex_ptr_dev() const { return ex_ptr_.empty() ? nullptr : d_ex_ptr_.as<int>(); }
    const int* ex_idx_dev() const { return ex_idx_.empty() ? nullptr : d_ex_idx_.as<int>(); }
    const int* sp_ptr_dev() const { return sp_ptr_.empty() ? nullptr : d_sp_ptr_.as<int>(); }
    const int* sp_idx_dev() const { return sp_idx_.empty() ? nullptr : d_sp_idx_.as<int>(); }

    // ------------------------------------------------------------------------------------------
    // geometry / capacity selection for the brick path
    int choose_geometry() {
        Geom<T>& g = g_;
        memset(&g, 0, sizeof(g));
        g.n = (int)n_;
        g.h = 2;
        g.align = 16 / (int)sizeof(T2);
        double vol = 1;
        for (int d = 0; d < 3; d++) {
            g.L[d] = (T)box_[d];
            g.invL[d] = (T)(1.0 / box_[d]);
            g.Ld[d] = box_[d];
            int nc = (int)std::floor(2.0 * box_[d] / r_list_);
            nc = std::max(nc, 5);
            while (nc > 5 && box_[d] / nc < 0.5 * r_list_ * (1.0 + 1e-6)) nc--;
            g.nc[d] = nc;
            g.celld[d] = box_[d] / nc;
            g.inv_cell[d] = (T)(nc / box_[d]);
            vol *= box_[d];
        }
        if ((double)g.nc[0] * g.nc[1] * g.nc[2] > 2.0e8) return set_error(MB_ERR_INVALID, "cell grid too large");
        if (dc_.nranks_ > g.nc[2]) return set_error(MB_ERR_INVALID, "more ranks than cell layers along z");
        g.ncells = g.nc[0] * g.nc[1] * g.nc[2];
        g.rlist2 = (T)(r_list_ * r_list_);
        g.skin_half2 = (T)(0.25 * skin_ * skin_);
        const double rho_c = (double)n_ / g.ncells;
        const double bytes_per_atom = sizeof(T4) + (P_.uniform_lj ? 0 : sizeof(T2));
        const double smem_budget = (double)smem_optin_ - 4096;
        int best[3] = {1, 1, 1};
        if (user_b_[0] > 0 && user_b_[1] > 0 && user_b_[2] > 0) {
            for (int d = 0; d < 3; d++) best[d] = std::min(user_b_[d], g.nc[d]);
            if (dc_.nranks_ > 1) best[2] = 1;
        } else {
            // Cost model in pair-evaluation units. The persistent force kernel keeps two CTAs per SM busy through a ring of
            // stages (one stage = one brick's halo), so a brick costs its pair work plus a staging share per halo atom and a
            // fixed hand-over cost; smaller bricks balance better across the 2 x n_sm CTAs (dynamic tickets), larger ones
            // stage fewer halo atoms per owned atom. The stage must leave room for at least two of them per CTA.
            const double nbrs = 4.18879 * r_list_ * r_list_ * r_list_ * (double)n_ / vol;
            const double cta_budget = ((double)smem_optin_ + 1024.0) / 2.0 - 3072.0;  // two CTAs share an SM's 228 KB
            const double slots = 2.0 * sm_count_;
            double best_t = 1e300;
            for (int bx = 1; bx <= 8; bx++)
                for (int by = 1; by <= bx; by++)
                    for (int bz = 1; bz <= by; bz++) {
                        if (bx > g.nc[0] || by > g.nc[1] || bz > g.nc[2]) continue;
                        if (dc_.nranks_ > 1 && bz != 1) continue;  // slabs are whole cell layers
                        double halo = (bx + 4.0) * (by + 4.0) * (bz + 4.0) * rho_c * 1.25 + 64;
                        double owned = (double)bx * by * bz * rho_c;
                        double smem = halo * bytes_per_atom + owned * 1.3 * 8.0 + 256;
                        if (smem > smem_budget || halo * 1.1 + 96 > LIST_MAX_HALO) continue;
                        const int stages2 = (int)std::floor(cta_budget / smem);  // ring depth with two CTAs per SM
                        double eff = stages2 >= 2 ? 1.0 : (stages2 == 1 ? 0.8 : 0.5);
                        // a stage hands out owned/4 quads to 15 consumer warps: with fewer than ~15 quads in flight over the
                        // ring the warps wait for the producer
                        eff *= std::min(1.0, std::max(1, std::min(stages2, 3)) * (owned / 4.0) / 15.0);
                        double cost_b = owned * nbrs + 6.0 * halo + 2000.0;
                        double nbr = std::ceil((double)g.nc[0] / bx) * std::ceil((double)g.nc[1] / by) * std::ceil((double)g.nc[2] / bz);
                        double t = (std::max(nbr / slots, 1.0) + 1.5) * cost_b / eff;  // + start-up and tail: about a brick and a half
                        if (t < best_t * 0.999) { best_t = t; best[0] = bx; best[1] = by; best[2] = bz; }
                    }
        }
        for (int d = 0; d < 3; d++) {
            g.b[d] = best[d];
            g.nb[d] = (g.nc[d] + g.b[d] - 1) / g.b[d];
            g.H[d] = g.b[d] + 2 * g.h;
        }
        g.nbricks = g.nb[0] * g.nb[1] * g.nb[2];
        for (int d = 0; d < 3; d++) g.nce[d] = g.nc[d] + 2 * g.h;
        g.necells = g.nce[0] * g.nce[1] * g.nce[2];
        g.nerows = g.nce[1] * g.nce[2];
        g.max_runs = g.H[1] * g.H[2];
        g.hcells = g.H[0] * g.H[1] * g.H[2];
        g.n_irows = g.b[1] * g.b[2];
        return MB_OK;
    }

    ExtMap<T> ext_map() const {
        ExtMap<T> m;
        m.ext_of = d_ext_of_.as<int>();
        m.gptr = d_gptr_.as<unsigned int>();
        m.ghosts = d_ghosts_.as<int2>();
        m.pos4e = (path_ == 1) ? d_pos4e_.as<T4>() : nullptr;
        for (int d = 0; d < 3; d++) m.Ld[d] = box_[d];
        return m;
    }
    // pos4e <- pos4 for slots [s0, s0 + n) (positions changed outside K1 and outside a rebuild)
    int ext_fill(int s0, int n) {
        if (n <= 0) return MB_OK;
        ext_fill_kernel<T><<<(n + 255) / 256, 256, 0, stream_>>>(ext_map(), s0, n, d_pos4_.as<T4>());
        launches_++;
        MB_CUDA(cudaGetLastError());
        return MB_OK;
    }
    size_t force_stage() const { return force_stage_bytes<T>(g_.halo_cap, g_.task_cap, P_.uniform_lj != 0); }
    // launch shape of the persistent force kernel: ring depth and CTAs per SM from the stage size. Two CTAs per SM when at
    // least one stage each fits (the f64 variants hold 128 registers per thread: one CTA), up to FORCE_MAX_STAGES stages.
    void force_shape(int& nbuf, int& ctas_per_sm) const {
        const size_t stage = force_stage();
        const size_t sm_total = smem_optin_ + 1024;  // 228 KB per SM, 1 KB reserved per resident CTA
        const size_t static_bytes = 1024;
        ctas_per_sm = (sizeof(T) == 8) ? 1 : FORCE_CTAS_F32;
        while (ctas_per_sm > 1 && (sm_total / ctas_per_sm - 1024 - static_bytes) / stage < 1) ctas_per_sm--;
        const size_t budget = (ctas_per_sm > 1) ? sm_total / ctas_per_sm - 1024 - static_bytes : smem_optin_ - static_bytes;
        nbuf = (int)std::min<size_t>(FORCE_MAX_STAGES, std::max<size_t>(1, budget / stage));
        nbuf = std::max(1, std::min(nbuf, env_.max_nbuf));  // MOLLYB200_NBUF: shallower ring
    }
    size_t build_smem_bytes() const {
        return (size_t)g_.halo_cap * (sizeof(T4) + sizeof(int)) + (size_t)((g_.hcells + 3) & ~3) * sizeof(ushort2) +
               (size_t)g_.n_irows * sizeof(IRow);
    }

    int alloc_brick_tables() {
        const Geom<T>& g = g_;
        MB_CUDA(d_cid_.ensure((size_t)(n_ + 16) * sizeof(int)));
        MB_CUDA(d_perm_.ensure((size_t)(n_ + 16) * sizeof(int)));
        MB_CUDA(d_cell_count_.ensure((size_t)(g.ncells + 2) * sizeof(int)));
        MB_CUDA(d_cell_start_.ensure((size_t)(g.ncells + 2) * sizeof(int)));
        MB_CUDA(d_cell_fill_.ensure((size_t)(g.ncells + 2) * sizeof(int)));
        MB_CUDA(cudaMemsetAsync(d_cell_count_.p, 0, (size_t)(g.ncells + 2) * sizeof(int), stream_));
        MB_CUDA(d_erow_total_.ensure((size_t)(g.nerows + 2) * sizeof(int)));
        MB_CUDA(d_erow_start_.ensure((size_t)(g.nerows + 2) * sizeof(int)));
        MB_CUDA(d_erow_fill_.ensure((size_t)(g.nerows + 2) * sizeof(int)));
        MB_CUDA(d_ecell_start_.ensure((size_t)(g.necells + 2) * sizeof(int)));
        MB_CUDA(d_ext_of_.ensure((size_t)(n_ + 16) * sizeof(int)));
        MB_CUDA(d_gptr_.ensure((size_t)(n_ + 16) * sizeof(unsigned int)));
        MB_CUDA(d_hdrs_.ensure((size_t)g.nbricks * sizeof(BrickHdr)));
        MB_CUDA(d_runs_.ensure((size_t)g.nbricks * g.max_runs * sizeof(Run)));
        MB_CUDA(d_irows_.ensure((size_t)g.nbricks * g.n_irows * sizeof(IRow)));
        MB_CUDA(d_hcs_.ensure((size_t)g.nbricks * g.hcells * sizeof(ushort2)));
        MB_CUDA(d_counts_.ensure((size_t)(n_ + 16) * sizeof(ushort2)));
        const size_t np = (size_t)n_ + 16;
        MB_CUDA(d_pos4_t_.ensure(np * sizeof(T4)));
        MB_CUDA(d_vel4_t_.ensure(np * sizeof(T4)));
        MB_CUDA(d_lj2_t_.ensure(np * sizeof(T2)));
        MB_CUDA(d_orig_t_.ensure(np * sizeof(int)));
        MB_CUDA(d_mass_t_.ensure(np * sizeof(T)));
        MB_CUDA(d_pe_partial_.ensure((size_t)std::max(std::max(g.nbricks, 4 * sm_count_), 1) * 7 * sizeof(double)));
        if (!d_sched_.p) {
            MB_CUDA(d_sched_.ensure(4 * sizeof(unsigned int)));
            MB_CUDA(cudaMemsetAsync(d_sched_.p, 0, 4 * sizeof(unsigned int), stream_));
        }
        return MB_OK;
    }

    // ---- terms added after the pair kernel: bonded lists and PME (specific.cuh, pme_host.cuh) ----------------------
    int set_specific(int kind, int64_t n, const int32_t* idx, const double* par) override {
        MB_TRY(bonded_.set(kind, n, idx, par, n_));
        destroy_graph();  // the step graph bakes the term counts in
        return MB_OK;
    }
    int set_pme(double r_cut, double error_tol, int order, double eps_r, int64_t n_pairs, const int32_t* pi, const int32_t* pj) override {
        MB_TRY(pme_.set(r_cut, error_tol, order, eps_r, n_pairs, pi, pj, n_));
        if (pme_.on_) destroy_graph();  // the captured step does not contain the PME launches
        return MB_OK;
    }
    int set_dispersion(double r_cut) override { return disp_.set(r_cut); }
    bool has_specific() const { return bonded_.any() || pme_.on_; }  // everything that is added after the pair kernel
    // add the bonded and PME forces to f4 (slot order on the brick path, original order on the all-pairs path);
    // with energy: their sum goes to bonded_.energy() (double, device)
    int launch_bonded(bool energy) {
        if (!has_specific()) return MB_OK;
        const int* slot_of = (path_ == 1) ? d_inv_orig_.as<int>() : nullptr;
        MB_TRY(bonded_.launch(energy, slot_of, d_pos4_.as<T4>(), d_f4_.as<T4>(), box_, launches_));
        if (pme_.on_)
            MB_TRY(pme_.launch(energy, n_, box_, h_charge_, d_pos4_.as<T4>(), d_f4_.as<T4>(), slot_of, bonded_.energy(), launches_));
        return MB_OK;
    }

    int comm_init(const void* uid, int rank, int nranks) override {
        MB_TRY(dc_.comm_init(uid, rank, nranks));
        have_list_ = false;
        dirty_ = true;
        return MB_OK;
    }

    // launch the list builder (count-only or real; with or without exclusion handling)
    int launch_build(bool count_only) {
        const size_t smem = build_smem_bytes();
        const bool has_ex = !ex_ptr_.empty() || !sp_ptr_.empty();
        MB_TRY(dispatch(count_only, [&](auto COUNT) {
            return dispatch(has_ex, [&](auto EX) -> int {
                auto kern = build_lists_kernel<T, COUNT, EX>;
                MB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                // few bricks (small systems, narrow slabs): several CTAs share a brick's atoms so that the SMs are filled
                const int nbr = dc_.own_nbricks(g_.nbricks);
                const int split = std::max(1, std::min(4, (4 * sm_count_ + nbr - 1) / std::max(nbr, 1)));
                kern<<<nbr * split, 256, smem, stream_>>>(d_ctl_.as<Control>(), g_, d_hdrs_.as<BrickHdr>(), d_runs_.as<Run>(),
                                                          d_irows_.as<IRow>(), d_hcs_.as<ushort2>(), d_pos4e_.as<T4>(), d_orig_e_.as<int>(),
                                                          ex_ptr_dev(), ex_idx_dev(), sp_ptr_dev(), sp_idx_dev(),
                                                          count_only ? nullptr : d_list_.as<unsigned short>(),
                                                          count_only ? nullptr : d_slist_.as<unsigned short>(),
                                                          count_only ? nullptr : d_counts_.as<ushort2>(),
                                                          count_only ? nullptr : d_task_tab_.as<int2>(), dc_.own_brick0(), split);
                return MB_OK;
            });
        }));
        launches_++;
        MB_CUDA(cudaGetLastError());
        return MB_OK;
    }

    // enqueue the gated rebuild sequence. count_only: first pass of the capacity derivation.
    int enqueue_rebuild(bool lists, bool count_only) {
        const Geom<T>& g = g_;
        Control* ctl = d_ctl_.as<Control>();
        const int nb = (int)((n_ + 255) / 256);
        prof_.begin(Prof::REBUILD);
        rebuild_begin_kernel<<<1, 32, 0, stream_>>>(ctl);
        bin_count_kernel<T><<<nb, 256, 0, stream_>>>(ctl, g, d_pos4_.as<T4>(), d_cid_.as<int>(), d_cell_count_.as<int>());
        cell_scan_kernel<<<1, 1024, 0, stream_>>>(ctl, g.ncells, g.n, d_cell_count_.as<int>(), d_cell_start_.as<int>(),
                                                  d_cell_fill_.as<int>());
        cell_scatter_kernel<<<nb, 256, 0, stream_>>>(ctl, g.n, d_cid_.as<int>(), d_cell_start_.as<int>(),
                                                     d_cell_fill_.as<int>(), d_perm_.as<int>());
        cell_sort_kernel<<<(g.ncells + 127) / 128, 128, 0, stream_>>>(ctl, g.ncells, d_cell_start_.as<int>(),
                                                                     d_perm_.as<int>(), d_cell_count_.as<int>());
        permute_gather_kernel<T><<<nb, 256, 0, stream_>>>(ctl, g.n, d_perm_.as<int>(), d_pos4_.as<T4>(), d_vel4_.as<T4>(),
                                                         d_lj2_.as<T2>(), d_orig_.as<int>(), d_mass_.as<T>(),
                                                         d_pos4_t_.as<T4>(), d_vel4_t_.as<T4>(), d_lj2_t_.as<T2>(),
                                                         d_orig_t_.as<int>(), d_mass_t_.as<T>());
        permute_commit_kernel<T><<<nb, 256, 0, stream_>>>(ctl, g.n, d_pos4_t_.as<T4>(), d_vel4_t_.as<T4>(), d_lj2_t_.as<T2>(),
                                                         d_orig_t_.as<int>(), d_mass_t_.as<T>(), d_pos4_.as<T4>(),
                                                         d_vel4_.as<T4>(), d_lj2_.as<T2>(), d_orig_.as<int>(), d_mass_.as<T>(),
                                                         d_xref4_.as<T4>(), d_inv_orig_.as<int>());
        // extended (ghost-padded) grid: row totals -> row starts (scan) -> cell starts -> per-atom map + ghost copies
        ext_row_totals_kernel<T><<<(g.nerows + 255) / 256, 256, 0, stream_>>>(ctl, g, d_cell_start_.as<int>(), d_erow_total_.as<int>());
        cell_scan_kernel<<<1, 1024, 0, stream_>>>(ctl, g.nerows, -1, d_erow_total_.as<int>(), d_erow_start_.as<int>(),
                                                  d_erow_fill_.as<int>());
        ext_cells_kernel<T><<<(g.necells + 1 + 255) / 256, 256, 0, stream_>>>(ctl, g, d_cell_start_.as<int>(), d_erow_start_.as<int>(),
                                                                            d_ecell_start_.as<int>());
        ext_atoms_kernel<T><<<nb, 256, 0, stream_>>>(ctl, g, d_cell_start_.as<int>(), d_ecell_start_.as<int>(), d_pos4_.as<T4>(),
                                                     P_.uniform_lj ? nullptr : d_lj2_.as<T2>(), d_ext_of_.as<int>(),
                                                     d_gptr_.as<unsigned int>(), d_ghosts_.as<int2>(), d_pos4e_.as<T4>(),
                                                     P_.uniform_lj ? nullptr : d_lj2e_.as<T2>(), d_orig_.as<int>(),
                                                     (ex_ptr_.empty() && sp_ptr_.empty()) ? nullptr : d_orig_e_.as<int>());
        brick_tables_kernel<T><<<g.nbricks, 128, 2 * g.max_runs * sizeof(int), stream_>>>(
            ctl, g, d_cell_start_.as<int>(), d_ecell_start_.as<int>(), d_hdrs_.as<BrickHdr>(), d_runs_.as<Run>(), d_irows_.as<IRow>(),
            d_hcs_.as<ushort2>(), g.task_cap > 0 ? d_task_tab_.as<int2>() : nullptr, P_.uniform_lj);
        launches_ += 12;
        if (lists) MB_TRY(launch_build(count_only));
        if (!count_only) {
            rebuild_finish_kernel<<<1, 32, 0, stream_>>>(ctl);
            launches_ += 1;
        }
        prof_.end(Prof::REBUILD);
        MB_CUDA(cudaGetLastError());
        return MB_OK;
    }

    // slot-order state in original order from coords (and the charges, LJ parts and masses of prepare())
    void init_slots(const T* coords_dev) {
        init_slots_kernel<T><<<(int)((n_ + 255) / 256), 256, 0, stream_>>>((int)n_, coords_dev, d_charge_in_.as<T>(), d_ljp_in_.as<T2>(),
                                                                        d_mass_in_.as<T>(), d_pos4_.as<T4>(), d_vel4_.as<T4>(),
                                                                        d_lj2_.as<T2>(), d_orig_.as<int>(), d_inv_orig_.as<int>(),
                                                                        d_mass_.as<T>(), d_xref4_.as<T4>());
        launches_++;
    }
    int read_ctl(Control& c) {
        MB_CUDA(cudaMemcpyAsync(&c, d_ctl_.p, sizeof(Control), cudaMemcpyDeviceToHost, stream_));
        MB_CUDA(cudaStreamSynchronize(stream_));
        return MB_OK;
    }
    int set_flag_rebuild() {
        static const int one = 1;
        MB_CUDA(cudaMemcpyAsync(&d_ctl_.as<Control>()->rebuild, &one, sizeof(int), cudaMemcpyHostToDevice, stream_));
        return MB_OK;
    }

    // Synchronous first build: derives halo capacity and list stride from the actual configuration.
    // coords_dev: n x 3 device array in original order.
    int first_build(const T* coords_dev) {
        dc_.build_nb_ = -1;  // lists for every brick (capacities are global; mb_forces evaluates the whole box)
        dc_.own_valid_ = false;
        init_slots(coords_dev);
        for (int attempt = 0; attempt < 8; attempt++) {
            MB_TRY(choose_geometry());
            MB_TRY(alloc_brick_tables());
            // pass A: sort + tables with unlimited halo capacity to measure
            g_.halo_cap = 65535;
            g_.stride = g_.sstride = g_.task_cap = g_.ext_cap = g_.ghost_cap = 0;
            MB_TRY(set_flag_rebuild());
            MB_TRY(enqueue_rebuild(false, true));
            Control c;
            MB_TRY(read_ctl(c));
            int cap = (int)(c.max_halo * (1.0 + 0.08 * cap_scale_)) + 32;  // temporal drift of the fullest brick's halo
            cap = (cap + 63) & ~63;
            g_.halo_cap = std::min(cap, LIST_MAX_HALO);
            g_.task_cap = (((int)(c.max_icount * (1.0 + 0.08 * cap_scale_)) + 8) + 1) & ~1;  // even: 16-byte rows for the bulk copy
            MB_CUDA(d_task_tab_.ensure((size_t)g_.nbricks * g_.task_cap * sizeof(int2)));
            // extended array / ghost table: measured sizes plus room for the boundary cells' population to drift
            g_.ext_cap = (int)std::min<double>(2.0e9, c.n_ext + (c.n_ext - (double)n_) * 0.10 * cap_scale_ + 1024);
            g_.ghost_cap = (int)std::min<double>(2.6e8, c.n_ghost * (1.0 + 0.10 * cap_scale_) + 1024);
            MB_CUDA(d_pos4e_.ensure(((size_t)g_.ext_cap + 64) * sizeof(T4)));
            MB_CUDA(cudaMemsetAsync(d_pos4e_.p, 0, ((size_t)g_.ext_cap + 64) * sizeof(T4), stream_));
            if (!P_.uniform_lj) {
                MB_CUDA(d_lj2e_.ensure(((size_t)g_.ext_cap + 64) * sizeof(T2)));
                MB_CUDA(cudaMemsetAsync(d_lj2e_.p, 0, ((size_t)g_.ext_cap + 64) * sizeof(T2), stream_));
            }
            if (!(ex_ptr_.empty() && sp_ptr_.empty())) MB_CUDA(d_orig_e_.ensure(((size_t)g_.ext_cap + 64) * sizeof(int)));
            MB_CUDA(d_ghosts_.ensure(((size_t)g_.ghost_cap + 64) * sizeof(int2)));
            size_t need = std::max(force_stage() + 2048, build_smem_bytes() + 1024);
            if (cap > LIST_MAX_HALO || need > smem_optin_) {  // list entries are 16-bit byte offsets of float4 records
                // shrink the brick and retry
                int* ub = user_b_;
                int cur[3] = {g_.b[0], g_.b[1], g_.b[2]};
                int dmax = 0;
                for (int d = 1; d < 3; d++) if (cur[d] > cur[dmax]) dmax = d;
                if (cur[dmax] == 1) return set_error(MB_ERR_CAPACITY, "halo of a single cell does not fit in shared memory (density too high for r_list)");
                cur[dmax]--;
                for (int d = 0; d < 3; d++) ub[d] = cur[d];
                continue;
            }
            // pass B: the pipeline again (idempotent: the positions are sorted) now that the extended array exists, with the
            // list builder only counting neighbours (the rebuild flag is still set because finish did not run)
            MB_TRY(enqueue_rebuild(true, true));
            MB_TRY(read_ctl(c));
            int stride = (int)(c.max_neighbors * (1.0 + 0.10 * cap_scale_)) + 16;
            stride = (stride + 31) & ~31;
            g_.stride = std::max(stride, 32);
            g_.sstride = std::max(8, (std::max(c.max_special, max_special_host_) + 7) & ~7);
            if (g_.stride > TASK_MAX_MAIN || g_.sstride > TASK_MAX_SPECIAL)
                return set_error(MB_ERR_CAPACITY, "neighbour rows longer than 4095 entries (or more than 255 special partners) are not supported");
            MB_CUDA(d_list_.ensure((size_t)(n_ + 16) * g_.stride * sizeof(unsigned short)));
            MB_CUDA(d_slist_.ensure((size_t)(n_ + 16) * g_.sstride * sizeof(unsigned short)));
            // pass C: the real build. The positions are already sorted; the pipeline is idempotent.
            MB_TRY(enqueue_rebuild(true, false));
            MB_TRY(read_ctl(c));
            if (c.overflow) return set_error(MB_ERR_CAPACITY, "neighbour capacity overflow during first build");
            have_list_ = true;
            geom_version_++;
            if (dc_.decomposed()) {
                MB_TRY(dc_.update_ownership(g_, d_cell_start_.as<int>()));
                dc_.since_rebuild_ = 0;
            }
            return MB_OK;
        }
        return set_error(MB_ERR_CAPACITY, "could not find a brick size that fits in shared memory");
    }

    // ------------------------------------------------------------------------------------------
    // the brick force kernel `kern` (one variant of brick_force_kernel) over bricks [brick0, brick0 + nbr)
    template <typename K>
    int launch_brick_force(K kern, ForceOut<T> out, int brick0, int nbr) {
        int nbuf, per_sm;
        force_shape(nbuf, per_sm);
        const size_t smem = (size_t)nbuf * force_stage();
        const int grid = std::max(1, std::min(nbr, per_sm * sm_count_));
        force_grid_ = grid;
        MB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        prof_.begin(Prof::FORCE);
        kern<<<grid, FORCE_THREADS, smem, stream_>>>(g_, P_, d_hdrs_.as<BrickHdr>(), d_runs_.as<Run>(), d_task_tab_.as<int2>(),
                                                     d_pos4e_.as<T4>(), d_lj2e_.as<T2>(), d_list_.as<unsigned short>(),
                                                     d_slist_.as<unsigned short>(), out, brick0, nbr, nbuf,
                                                     env_.static_sched ? nullptr : d_sched_.as<unsigned int>());
        prof_.end(Prof::FORCE);
        launches_++;
        n_force_evals_++;
        MB_CUDA(cudaGetLastError());
        return MB_OK;
    }
    // owned_only: in a decomposed run the step loop evaluates only this rank's slab of bricks
    int launch_force(bool energy, bool owned_only = false) {
        const int b0 = owned_only ? dc_.own_b0_ : 0;
        const int nbr = owned_only ? dc_.own_nb_ : g_.nbricks;
        ForceOut<T> out;
        out.f4 = d_f4_.as<T4>();
        out.pe_partial = d_pe_partial_.as<double>();
        out.vir_partial = d_pe_partial_.as<double>() + std::max(g_.nbricks, 4 * sm_count_);
        out.gate = dc_.gate_;  // one-shot: set by the decomposed step in front of this launch
        memset(&dc_.gate_, 0, sizeof(dc_.gate_));
        return dispatch(BrickCoulKinds{}, P_.coul_kind, [&](auto COUL) {
            return dispatch(BrickCutModes{}, cutm_, [&](auto CUTM) {
                return dispatch(energy, [&](auto EN) {
                    if constexpr (COUL == COUL_NONE)
                        return dispatch(P_.uniform_lj != 0, [&](auto UNI) {
                            return launch_brick_force(brick_force_kernel<T, COUL, UNI, CUTM, EN>, out, b0, nbr);
                        });
                    else
                        return launch_brick_force(brick_force_kernel<T, COUL, false, CUTM, EN>, out, b0, nbr);
                });
            }, "experiment build: plain cutoffs only");
        }, "experiment build: LJ and LJ + CoulombReactionField only");
    }

    // no-list kernel over pos4 / lj2 in original order, forces into f4
    int launch_allpairs(bool energy) {
        const int nblk = (int)((n_ + AP_THREADS - 1) / AP_THREADS);
        MB_CUDA(d_pe_partial_.ensure((size_t)nblk * 7 * sizeof(double)));
        double* pe = d_pe_partial_.as<double>();
        double* vir = pe + nblk;
        T Lx = (T)box_[0], Ly = (T)box_[1], Lz = (T)box_[2];
        prof_.begin(Prof::FORCE);
        MB_TRY(dispatch(AllCoulKinds{}, P_.coul_kind, [&](auto COUL) {
            return dispatch(AllCutModes{}, cutm_, [&](auto CUTM) {
                return dispatch(energy, [&](auto EN) {
                    allpairs_force_kernel<T, COUL, CUTM, EN><<<nblk, AP_THREADS, 0, stream_>>>(
                        (int)n_, P_, Lx, Ly, Lz, tric_, d_pos4_.as<T4>(), d_lj2_.as<T2>(), ex_ptr_dev(), ex_idx_dev(), sp_ptr_dev(), sp_idx_dev(),
                        d_f4_.as<T4>(), pe, vir);
                    return MB_OK;
                });
            });
        }));
        prof_.end(Prof::FORCE);
        launches_++;
        n_force_evals_++;
        MB_CUDA(cudaGetLastError());
        return MB_OK;
    }

    // host/device argument views ----------------------------------------------------------------
    // device pointer for `count` T outputs to `user`: user itself if it is device memory, else the staging buffer, which
    // view_out_done copies back; `load` fills the stage with user's values first (in-out arguments, outputs added to)
    int view_out(void* user, size_t count, DevBuf& stage, bool load, T** out) {
        if (!user || is_device_ptr(user)) { *out = reinterpret_cast<T*>(user); return MB_OK; }
        MB_CUDA(stage.ensure(count * sizeof(T)));
        if (load) MB_CUDA(cudaMemcpyAsync(stage.p, user, count * sizeof(T), cudaMemcpyHostToDevice, stream_));
        *out = stage.as<T>();
        return MB_OK;
    }
    int view_out_done(void* user, const T* dev, size_t count) {
        if (dev != user) MB_CUDA(cudaMemcpyAsync(user, dev, count * sizeof(T), cudaMemcpyDeviceToHost, stream_));
        return MB_OK;
    }
    // device pointer holding `count` T values of `user` (copied if user is a host pointer)
    int view_in(const void* user, size_t count, DevBuf& stage, const T** out) {
        T* p = nullptr;
        MB_TRY(view_out(const_cast<void*>(user), count, stage, true, &p));
        *out = p;
        return MB_OK;
    }
    // per-block partial sums of a velocity reduction (kern writes k doubles per 256-thread block) -> s[0..k) on the host
    int reduce_to_host(void (*kern)(int, const T*, const T*, double*), const T* vels, int k, double* s) {
        const int nb = (int)((n_ + 255) / 256);
        MB_CUDA(d_partial_.ensure((size_t)nb * k * sizeof(double)));
        kern<<<nb, 256, 0, stream_>>>((int)n_, vels, d_mass_in_.as<T>(), d_partial_.as<double>());
        launches_++;
        std::vector<double> part((size_t)nb * k);
        MB_CUDA(cudaMemcpyAsync(part.data(), d_partial_.p, part.size() * sizeof(double), cudaMemcpyDeviceToHost, stream_));
        MB_CUDA(cudaStreamSynchronize(stream_));
        for (int d = 0; d < k; d++) s[d] = 0;
        for (int b = 0; b < nb; b++) for (int d = 0; d < k; d++) s[d] += part[(size_t)k * b + d];
        return MB_OK;
    }

    // ------------------------------------------------------------------------------------------
    // make the slot-order state reflect `coords` (and vels), rebuilding the list when required
    int sync_state_from(const T* coords_dev, const T* vels_dev) {
        const bool first = !have_list_;
        if (first) MB_TRY(first_build(coords_dev));
        if (first && !vels_dev) return MB_OK;
        // right after a first build the displacement check reports into ctl->disp instead of requesting a rebuild
        ingest_kernel<T><<<(int)((n_ + 255) / 256), 256, 0, stream_>>>((int)n_, g_, coords_dev, vels_dev, d_orig_.as<int>(),
                                                                    d_xref4_.as<T4>(), d_pos4_.as<T4>(), d_vel4_.as<T4>(),
                                                                    first ? &d_ctl_.as<Control>()->disp : &d_ctl_.as<Control>()->rebuild);
        launches_++;
        if (first) return ext_fill(0, (int)n_);
        if (dc_.decomposed()) {
            // Every rank holds the full state here. The lists of the previous call stay valid until an atom has moved more
            // than skin/2 from its position at the last rebuild (ingest_kernel just checked that on identical data on every
            // rank) or the rebuild interval has run out; the host needs the answer because ownership follows from the sort.
            int flag = 0;
            MB_CUDA(cudaMemcpyAsync(&flag, &d_ctl_.as<Control>()->rebuild, sizeof(int), cudaMemcpyDeviceToHost, stream_));
            MB_CUDA(cudaStreamSynchronize(stream_));
            if (flag || !dc_.own_valid_ || dc_.since_rebuild_ >= dc_.interval(rebuild_every_)) {
                if (dc_.own_valid_) { dc_.build_b0_ = dc_.own_b0_; dc_.build_nb_ = dc_.own_nb_; }  // lists only for the owned slab
                MB_TRY(set_flag_rebuild());
                MB_TRY(enqueue_rebuild(true, false));
                MB_TRY(dc_.update_ownership(g_, d_cell_start_.as<int>()));
                dc_.since_rebuild_ = 0;
            } else {
                MB_TRY(ext_fill(0, (int)n_));
            }
            return MB_OK;
        }
        MB_TRY(enqueue_rebuild(true, false));
        MB_TRY(ext_fill(0, (int)n_));  // (a rebuild refilled pos4e itself; without one the ingested positions go in here)
        return MB_OK;
    }

    // end of a call: on the brick path read back the capacity flags (a host wait), else just wait
    int finish_call() {
        MB_CUDA(cudaGetLastError());
        if (path_ == 0) {
            MB_CUDA(cudaStreamSynchronize(stream_));
            return MB_OK;
        }
        Control c;
        MB_TRY(read_ctl(c));
        if (c.overflow) {
            have_list_ = false;  // next call re-derives capacities
            static const int zero = 0;
            cudaMemcpyAsync(&d_ctl_.as<Control>()->overflow, &zero, sizeof(int), cudaMemcpyHostToDevice, stream_);
            return set_error(MB_ERR_CAPACITY, "neighbour/halo capacity overflow; results of this call are invalid, retry");
        }
        return MB_OK;
    }

    // ------------------------------------------------------------------------------------------
    int forces_energy(const void* coords, void* fs, void* pe, void* vir, int64_t step_n, bool with_specific) override {
        (void)step_n;
        MB_TRY(prepare());
        if (!coords) return set_error(MB_ERR_INVALID, "coords is null");
        const T* xc = nullptr;
        MB_TRY(view_in(coords, 3 * (size_t)n_, d_stage_a_, &xc));
        const bool energy = (pe != nullptr) || (vir != nullptr);
        const int nb = (int)((n_ + 255) / 256);
        int n_partials = 0;
        const int* orig = nullptr;
        if (path_ == 0) {
            init_slots(xc);  // original order; posq packed into pos4
            MB_TRY(launch_allpairs(energy));
            n_partials = (int)((n_ + AP_THREADS - 1) / AP_THREADS);
        } else {
            if (dc_.decomposed()) have_list_ = false;  // forces()/potential_energy() evaluate the whole box on every rank
            MB_TRY(sync_state_from(xc, nullptr));
            MB_TRY(launch_force(energy));
            n_partials = force_grid_;
            orig = d_orig_.as<int>();
        }
        if (with_specific) MB_TRY(launch_bonded(pe != nullptr));
        // outputs (ADD semantics)
        if (fs) {
            T* fo = nullptr;
            MB_TRY(view_out(fs, 3 * (size_t)n_, d_stage_b_, true, &fo));
            scatter_forces_kernel<T><<<nb, 256, 0, stream_>>>((int)n_, d_f4_.as<T4>(), orig, fo);
            launches_++;
            MB_TRY(view_out_done(fs, fo, 3 * (size_t)n_));
        }
        if (energy) {
            // stage scalars on device: [pe, vir(9)]
            MB_CUDA(d_scalars_.ensure(16 * sizeof(T)));
            T host_sc[16] = {0};
            bool pe_dev = pe && is_device_ptr(pe), vir_dev = vir && is_device_ptr(vir);
            T* pe_target = nullptr;
            T* vir_target = nullptr;
            if (pe) {
                if (pe_dev) pe_target = reinterpret_cast<T*>(pe);
                else { host_sc[0] = *reinterpret_cast<T*>(pe); pe_target = d_scalars_.as<T>(); }
            }
            if (vir) {
                if (vir_dev) vir_target = reinterpret_cast<T*>(vir);
                else { memcpy(host_sc + 1, vir, 9 * sizeof(T)); vir_target = d_scalars_.as<T>() + 1; }
            }
            if ((pe && !pe_dev) || (vir && !vir_dev))
                MB_CUDA(cudaMemcpyAsync(d_scalars_.p, host_sc, 16 * sizeof(T), cudaMemcpyHostToDevice, stream_));
            double* pp = d_pe_partial_.as<double>();
            const double* vp = (path_ == 1) ? pp + std::max(g_.nbricks, 4 * sm_count_) : pp + n_partials;
            reduce_partials_kernel<T><<<1, 256, 0, stream_>>>(n_partials, pp, vp, pe_target, vir_target, nullptr);
            launches_++;
            if (with_specific && has_specific() && pe_target) {
                add_double_kernel<T><<<1, 1, 0, stream_>>>(bonded_.energy(), pe_target);
                launches_++;
            }
            if (with_specific && disp_.rc_ > 0) {  // LJDispersionCorrection: E = (f6 + f12) / V; virial 2 U6 + 4 U12 on the diagonal
                MB_TRY(disp_.prepare(n_, h_sigma_, h_eps_raw_));
                const double vol = box_[0] * box_[1] * box_[2];
                const double u6 = disp_.f6_ / vol, u12 = disp_.f12_ / vol;
                add_scalars_kernel<T><<<1, 1, 0, stream_>>>(pe_target, (T)(u6 + u12), vir_target, (T)(2.0 * u6 + 4.0 * u12));
                launches_++;
            }
            if ((pe && !pe_dev) || (vir && !vir_dev)) {
                MB_CUDA(cudaMemcpyAsync(host_sc, d_scalars_.p, 16 * sizeof(T), cudaMemcpyDeviceToHost, stream_));
                MB_CUDA(cudaStreamSynchronize(stream_));
                if (pe && !pe_dev) *reinterpret_cast<T*>(pe) = host_sc[0];
                if (vir && !vir_dev) memcpy(vir, host_sc + 1, 9 * sizeof(T));
            }
        }
        return finish_call();
    }

    // ------------------------------------------------------------------------------------------
    // One MD step enqueued on the stream. In capture mode the neighbour rebuild becomes the body of a CUDA-graph
    // conditional node driven by decide_kernel, otherwise the gated pipeline is enqueued when it may be needed.
    struct StepCfg {
        T dt, dt_half, skin_half2, kT;
        double prob, inv_mass;
        int do_cm;        // 0/1 constant, or -1: caller decides per step (stream path only)
        bool thermostat;
        int* flag_ptr;
    };
    int enqueue_step(const StepCfg& c, int do_cm_now, bool clear_cm_after_k1, bool capture,
                     cudaGraphConditionalHandle handle, cudaGraph_t graph, cudaGraph_t* body_out, bool host_rebuild_hint,
                     bool defer_cm = false) {
        const bool dec = dc_.decomposed() && path_ == 1;
        const int s0 = dec ? dc_.own_s0_ : 0, n_own = dec ? dc_.own_n_ : (int)n_;
        const int nb = std::max(1, (n_own + 255) / 256);
        Control* ctl = d_ctl_.as<Control>();
        CmState<T>* cm = d_cm_.as<CmState<T>>();
        // decomposed run over peer memory (peer.cuh): K1 mirrors the boundary slots into the neighbours while it drifts
        const unsigned long long epoch = dec ? ++dc_.epoch_ : 0ull;
        const bool p2p_halo = dec && dc_.p2p_active() && !host_rebuild_hint;  // rebuild steps all-gather the state instead
        PeerPush<T> push;
        memset(&push, 0, sizeof(push));
        if (p2p_halo) push = dc_.make_push(epoch, true);
        if (dc_.cm_deferred_epoch_) {  // the previous step left v_cm in the momentum all-to-all (no peer_cm_kernel)
            push.cm_comm = dc_.comm_of(dc_.rank_);
            push.cm_nranks = dc_.nranks_;
            push.cm_epoch = dc_.cm_deferred_epoch_;
            push.cm_inv_mass = c.inv_mass;
            dc_.cm_deferred_epoch_ = 0;
        }
        prof_.begin(Prof::VV);
        const Thermo<T> th = thermo_in_k1(c);
        auto k1 = th.on ? vv_kick_drift_kernel<T, true> : vv_kick_drift_kernel<T, false>;
        k1<<<std::max(1, std::min((nb + 1) / 2, 5 * sm_count_)), 256, 0, stream_>>>(  // two atoms per thread, one wave (48 registers: 5 CTAs per SM)
            s0, n_own, c.dt, c.dt_half, c.skin_half2, cm, d_f4_.as<T4>(), d_xref4_.as<T4>(), d_pos4_.as<T4>(), d_vel4_.as<T4>(),
            c.flag_ptr, ctl, handle, capture && path_ == 1 ? 1 : 0, push, ext_map(), th);
        prof_.end(Prof::VV);
        launches_++;
        if (clear_cm_after_k1) {
            clear_cm_kernel<T><<<1, 1, 0, stream_>>>(cm);
            launches_++;
        }
        if (path_ == 0) {
            wrap_kernel<T><<<nb, 256, 0, stream_>>>((int)n_, g_ap_, d_pos4_.as<T4>());
            launches_++;
        } else if (capture) {
            // splice a conditional IF node into the capture; its body is filled in by the caller
            cudaStreamCaptureStatus status;
            const cudaGraphNode_t* deps = nullptr;
            size_t ndeps = 0;
            cudaGraph_t gcap = nullptr;
            MB_CUDA(cudaStreamGetCaptureInfo_v2(stream_, &status, nullptr, &gcap, &deps, &ndeps));
            cudaGraphNodeParams cp = {cudaGraphNodeTypeConditional};
            cp.type = cudaGraphNodeTypeConditional;
            cp.conditional.handle = handle;
            cp.conditional.type = cudaGraphCondTypeIf;
            cp.conditional.size = 1;
            cudaGraphNode_t cnode;
            MB_CUDA(cudaGraphAddNode(&cnode, graph, deps, ndeps, &cp));
            *body_out = cp.conditional.phGraph_out[0];
            MB_CUDA(cudaStreamUpdateCaptureDependencies(stream_, &cnode, 1, cudaStreamSetCaptureDependencies));
        } else if (dec) {
            if (host_rebuild_hint) {
                // neighbour rebuild on a decomposed box: replicate positions and velocities, rebuild (identical sort on every
                // rank, lists only for the owned slab), then refresh the slot ranges and halo segments
                MB_TRY(dc_.allgather_state(g_, d_pos4_.as<T4>(), d_vel4_.as<T4>()));
                MB_TRY(set_flag_rebuild());
                MB_TRY(enqueue_rebuild(true, false));
                MB_TRY(dc_.update_ownership(g_, d_cell_start_.as<int>()));
            } else if (p2p_halo) {
                dc_.gate_ = dc_.make_wait(epoch);  // the force kernel's CTAs wait for the neighbours' pushes of this epoch
            } else {
                MB_TRY(dc_.halo_exchange(d_pos4_.as<T4>()));
                for (auto& sg : dc_.halo_recv_) MB_TRY(ext_fill(sg.start, sg.count));  // received slots -> extended array (+ ghost copies)
            }
        } else {
            if (rebuild_every_ == 0 || host_rebuild_hint) MB_TRY(enqueue_rebuild(true, false));
        }
        const int s0b = dec ? dc_.own_s0_ : 0, n_ownb = dec ? dc_.own_n_ : (int)n_;  // ownership may have changed in the rebuild
        const int nb2 = std::max(1, (n_ownb + 255) / 256);
        const int vvb2 = std::max(1, std::min((n_ownb + 2 * VV_THREADS - 1) / (2 * VV_THREADS), 8 * sm_count_));
        if (path_ == 0) MB_TRY(launch_allpairs(false));
        else MB_TRY(launch_force(false, dec));
        MB_TRY(launch_bonded(false));
        const bool p2p_sig = dec && dc_.p2p_active();  // (after a rebuild: the new ownership's peers)
        PeerSignal sig;
        memset(&sig, 0, sizeof(sig));
        if (p2p_sig) sig = dc_.make_signal(epoch, do_cm_now != 0);
        prof_.begin(Prof::VV);
        vv_kick2_kernel<T><<<vvb2, VV_THREADS, 0, stream_>>>(s0b, n_ownb, c.dt_half, do_cm_now, c.inv_mass, d_f4_.as<T4>(), d_mass_.as<T>(),
                                                             d_vel4_.as<T4>(), d_partial_.as<double>(), ctl, cm, 0,
                                                             dec ? dc_.mom() : nullptr, sig);
        prof_.end(Prof::VV);
        launches_++;
        if (p2p_sig && do_cm_now && defer_cm && !c.thermostat) {
            dc_.cm_deferred_epoch_ = epoch;  // the next step's K1 adds the slabs' sums itself
        } else if (p2p_sig && do_cm_now) {
            // sum(m v) of all slabs arrived by peer stores: add them in rank order
            peer_cm_kernel<T><<<1, 32, 0, stream_>>>(dc_.comm_of(dc_.rank_), dc_.nranks_, epoch, c.inv_mass, cm);
            launches_++;
        } else if (dec && do_cm_now) {
            // global sum(m v): one 24-byte all-reduce per step, then v_cm for the lazy subtraction
            double* mom = dc_.mom();
            MB_NCCL(g_nccl.AllReduce(mom, mom + 4, 3, ncclDouble, ncclSum, dc_.comm_, stream_));
            cm_from_sum_kernel<T><<<1, 1, 0, stream_>>>(mom + 4, c.inv_mass, cm);
            launches_++;
        }
        if (c.thermostat && !thermo_in_k1(c).on) {
            andersen_kernel<T><<<nb2, 256, 0, stream_>>>(s0b, n_ownb, (int)n_, c.kT, c.prob, d_orig_.as<int>(), d_mass_.as<T>(), d_vel4_.as<T4>(), cm, ctl);
            launches_++;
        }
        MB_CUDA(cudaGetLastError());
        return MB_OK;
    }
    // single-GPU step loop: the thermostat of step n runs at the top of step n+1's drift kernel; the last step of a call is
    // closed by the standalone kernel (simulate_vv)
    Thermo<T> thermo_in_k1(const StepCfg& c) const {
        Thermo<T> th;
        memset(&th, 0, sizeof(th));
        if (c.thermostat && !dc_.decomposed()) {
            th.on = 1;
            th.n = (int)n_;
            th.kT = c.kT;
            th.prob = c.prob;
            th.orig = d_orig_.as<int>();
            th.mass = d_mass_.as<T>();
        }
        return th;
    }

    struct GraphKey {
        int path, do_cm, thermostat, geom_version, rebuild_every;
        double dt, kT, prob;
        int64_t n;
        bool operator==(const GraphKey& o) const {
            return path == o.path && do_cm == o.do_cm && thermostat == o.thermostat && geom_version == o.geom_version &&
                   rebuild_every == o.rebuild_every && dt == o.dt && kT == o.kT && prob == o.prob && n == o.n;
        }
    };
    void destroy_graph() {
        if (graph_exec_) cudaGraphExecDestroy(graph_exec_);
        if (graph_) cudaGraphDestroy(graph_);
        graph_exec_ = nullptr;
        graph_ = nullptr;
    }
    // Capture one MD step (K1, decide, [IF rebuild], force, K2, [thermostat]) into an executable graph.
    int build_step_graph(const StepCfg& c, const GraphKey& key) {
        destroy_graph();
        const bool prof_was = prof_.enabled;
        prof_.enabled = false;
        const int64_t launches_before = launches_;
        auto fail = [&](int rc) {
            cudaStreamCaptureStatus st;
            if (cudaStreamIsCapturing(stream_, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone) {
                cudaGraph_t junk = nullptr;
                cudaStreamEndCapture(stream_, &junk);
            }
            cudaGetLastError();
            destroy_graph();
            prof_.enabled = prof_was;
            launches_ = launches_before;
            return rc;
        };
        if (cudaGraphCreate(&graph_, 0) != cudaSuccess) return fail(MB_ERR_CUDA);
        cudaGraphConditionalHandle handle = 0;
        if (path_ == 1 && cudaGraphConditionalHandleCreate(&handle, graph_, 0, cudaGraphCondAssignDefault) != cudaSuccess)
            return fail(MB_ERR_CUDA);
        if (cudaStreamBeginCaptureToGraph(stream_, graph_, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed) != cudaSuccess)
            return fail(MB_ERR_CUDA);
        cudaGraph_t body = nullptr;
        if (enqueue_step(c, c.do_cm, false, true, handle, graph_, &body, false) != MB_OK) return fail(MB_ERR_CUDA);
        cudaGraph_t out = nullptr;
        if (cudaStreamEndCapture(stream_, &out) != cudaSuccess) return fail(MB_ERR_CUDA);
        const int64_t step_nodes = launches_ - launches_before;
        if (path_ == 1) {
            if (!body) return fail(MB_ERR_CUDA);
            if (cudaStreamBeginCaptureToGraph(stream_, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed) != cudaSuccess)
                return fail(MB_ERR_CUDA);
            if (enqueue_rebuild(true, false) != MB_OK) return fail(MB_ERR_CUDA);
            if (cudaStreamEndCapture(stream_, &out) != cudaSuccess) return fail(MB_ERR_CUDA);
        }
        if (cudaGraphInstantiate(&graph_exec_, graph_, 0) != cudaSuccess) return fail(MB_ERR_CUDA);
        prof_.enabled = prof_was;
        launches_ = launches_before;
        graph_step_launches_ = step_nodes;
        graph_key_ = key;
        return MB_OK;
    }

    int simulate_vv(void* coords, void* vels, const mb_vv_params_t* p) override {
        MB_TRY(prepare());
        if (!coords || !vels || !p) return set_error(MB_ERR_INVALID, "null argument");
        if (p->n_steps < 0 || !(p->dt > 0)) return set_error(MB_ERR_INVALID, "n_steps < 0 or dt <= 0");
        const T* xc = nullptr;
        const T* vc = nullptr;
        MB_TRY(view_in(coords, 3 * (size_t)n_, d_stage_a_, &xc));
        MB_TRY(view_in(vels, 3 * (size_t)n_, d_stage_c_, &vc));
        const int nb = (int)((n_ + 255) / 256);
        const int vvb = std::min((int)((n_ + VV_THREADS - 1) / VV_THREADS), 8 * sm_count_);
        Control* ctl = d_ctl_.as<Control>();
        CmState<T>* cm = d_cm_.as<CmState<T>>();
        clear_cm_kernel<T><<<1, 1, 0, stream_>>>(cm);
        launches_++;
        StepCfg c;
        c.dt = (T)p->dt;
        c.dt_half = (T)p->dt / (T)2;
        c.inv_mass = (total_mass_ > 0) ? 1.0 / total_mass_ : 0.0;
        c.thermostat = p->andersen_kT > 0 && p->andersen_prob > 0;
        c.kT = (T)p->andersen_kT;
        c.prob = p->andersen_prob;
        c.do_cm = (p->remove_cm_every == 0) ? 0 : (p->remove_cm_every == 1 ? 1 : -1);
        if (path_ == 0) {
            init_slots(xc);
            // velocities + wrap through ingest with an identity order (geometry only needs L)
            Geom<T> g0;
            memset(&g0, 0, sizeof(g0));
            for (int d = 0; d < 3; d++) { g0.L[d] = (T)box_[d]; g0.invL[d] = (T)(1.0 / box_[d]); }
            g0.skin_half2 = std::numeric_limits<T>::infinity();
            g0.tric = tric_;
            g_ap_ = g0;
            ingest_kernel<T><<<nb, 256, 0, stream_>>>((int)n_, g0, xc, vc, d_orig_.as<int>(), d_xref4_.as<T4>(), d_pos4_.as<T4>(),
                                                      d_vel4_.as<T4>(), &ctl->disp);
            wrap_kernel<T><<<nb, 256, 0, stream_>>>((int)n_, g0, d_pos4_.as<T4>());
            launches_ += 2;
            c.skin_half2 = std::numeric_limits<T>::infinity();
            c.flag_ptr = &ctl->disp;
        } else {
            MB_TRY(sync_state_from(xc, vc));
            c.skin_half2 = g_.skin_half2;  // geometry is chosen by the first build
            c.flag_ptr = (rebuild_every_ == 0 && !dc_.decomposed()) ? &ctl->rebuild : &ctl->disp;
        }
        // step bookkeeping lives on the device (tail of Control)
        {
            struct Tail { int rebuild_every; long long step, init_step; unsigned int rng[4]; unsigned int max_disp2_bits, call_max_disp2_bits; } t;
            static_assert(sizeof(Tail) == sizeof(Control) - offsetof(Control, rebuild_every), "Control tail layout");
            t.rebuild_every = (dc_.decomposed() && path_ == 1) ? 0 : rebuild_every_;  // decomposed: the host counts the interval
            t.step = p->init_step;
            t.init_step = p->init_step;
            t.rng[0] = (unsigned int)p->rng_ctr1; t.rng[1] = (unsigned int)(p->rng_ctr1 >> 32);
            t.rng[2] = (unsigned int)p->rng_key; t.rng[3] = (unsigned int)(p->rng_key >> 32);
            t.max_disp2_bits = 0;
            t.call_max_disp2_bits = 0;
            MB_CUDA(cudaMemcpyAsync(reinterpret_cast<char*>(ctl) + offsetof(Control, rebuild_every), &t, sizeof(t),
                                    cudaMemcpyHostToDevice, stream_));
            MB_CUDA(cudaStreamSynchronize(stream_));  // t is a local
        }
        dc_.cm_deferred_epoch_ = 0;
        dc_.adapt_span_ = dc_.since_rebuild_;
        bool cm_pending = false;  // host mirror of cm->valid
        if (p->init_step == 0 && p->remove_cm_every != 0) {
            // remove_CM_motion! before the first force evaluation (simulators.jl:563): zero-length kick
            vv_kick2_kernel<T><<<vvb, VV_THREADS, 0, stream_>>>(0, (int)n_, (T)0, 1, c.inv_mass, d_f4_.as<T4>(), d_mass_.as<T>(),
                                                                d_vel4_.as<T4>(), d_partial_.as<double>(), ctl, cm, 0, nullptr,
                                                                PeerSignal{});
            launches_++;
            cm_pending = true;
        }
        const bool dec = dc_.decomposed() && path_ == 1;
        if (dec && pme_.on_) return set_error(MB_ERR_INVALID, "PME is not available in decomposed (multi-GPU) runs yet");
        if (dec) {
            // lists built from here on cover only the owned slab
            dc_.build_b0_ = dc_.own_b0_;
            dc_.build_nb_ = dc_.own_nb_;
            MB_TRY(dc_.p2p_setup(d_pos4e_.p, env_.p2p));  // collective; falls back to the NCCL transport on every rank if any mapping fails
        }
        if (path_ == 0) MB_TRY(launch_allpairs(false));
        else MB_TRY(launch_force(false, dec));
        MB_TRY(launch_bonded(false));
        if (dec) {
            const unsigned long long e0 = ++dc_.epoch_;  // this force evaluation read the replicated state: tell the pushers
            if (dc_.p2p_active()) {
                peer_signal_kernel<<<1, 32, 0, stream_>>>(dc_.make_signal(e0, false));
                launches_++;
            }
        }

        // CUDA-graph path: static per-step sequence (remove_CM_motion in {0,1}, no stage timers requested)
        bool use_graph = env_.graph && !graph_failed_ && !prof_.enabled && c.do_cm >= 0 && p->n_steps >= 4 &&
                         !(cm_pending && c.do_cm == 0) && !dec &&  // the decomposed step issues NCCL calls with per-rebuild sizes
                         !pme_.on_;                                  // cuFFT launches stay outside the captured step for now
        if (use_graph) {
            GraphKey key{path_, c.do_cm, c.thermostat ? 1 : 0, geom_version_, rebuild_every_, p->dt, p->andersen_kT, p->andersen_prob, n_};
            if (!graph_exec_ || !(key == graph_key_)) {
                if (build_step_graph(c, key) != MB_OK) {
                    graph_failed_ = true;  // stay on the stream path for this context
                    use_graph = false;
                }
            }
        }
        graph_used_ = use_graph;
        if (use_graph) {
            for (int64_t k = 1; k <= p->n_steps; k++) MB_CUDA(cudaGraphLaunch(graph_exec_, stream_));
            launches_ += graph_step_launches_ * p->n_steps;  // rebuild-body kernels are not counted
            n_force_evals_ += p->n_steps;
            n_steps_ += p->n_steps;
        } else {
            for (int64_t k = 1; k <= p->n_steps; k++) {
                const int64_t step_n = p->init_step + k;
                const int do_cm = (p->remove_cm_every != 0 && step_n % p->remove_cm_every == 0) ? 1 : 0;
                const bool clear_after_k1 = cm_pending && !do_cm;  // K1 consumed v_cm; nothing overwrites it this step
                // decomposed: fixed interval counted on the host (identical on every rank), adapted per call from the displacements
                bool hint;
                if (dec) {
                    hint = dc_.since_rebuild_ >= dc_.interval(rebuild_every_);
                    dc_.since_rebuild_ = hint ? 1 : dc_.since_rebuild_ + 1;
                    dc_.adapt_span_ = std::max(dc_.adapt_span_, dc_.since_rebuild_);
                } else {
                    hint = rebuild_every_ > 0 && k > 1 && (step_n - 1) % rebuild_every_ == 0;
                }
                MB_TRY(enqueue_step(c, do_cm, clear_after_k1, false, 0, nullptr, nullptr, hint, /*defer_cm=*/k < p->n_steps));
                cm_pending = (do_cm != 0) && !(c.thermostat && dec);  // (the standalone thermostat kernel consumes v_cm)
                n_steps_++;
            }
        }
        if (c.thermostat && !dec && p->n_steps > 0) {
            // the thermostat of the last step (the earlier ones ran inside the next step's drift kernel)
            andersen_kernel<T><<<nb, 256, 0, stream_>>>(0, (int)n_, (int)n_, c.kT, c.prob, d_orig_.as<int>(), d_mass_.as<T>(), d_vel4_.as<T4>(), cm, ctl);
            launches_++;
        }
        if (dec) {
            MB_TRY(dc_.allgather_state(g_, d_pos4_.as<T4>(), d_vel4_.as<T4>()));  // every rank returns the whole system
            dc_.build_nb_ = -1;
            if (rebuild_every_ == 0) MB_TRY(dc_.adapt_interval(ctl, skin_, launches_));
        }
        // export
        T *xo = nullptr, *vo = nullptr;
        MB_TRY(view_out(coords, 3 * (size_t)n_, d_stage_a_, false, &xo));
        MB_TRY(view_out(vels, 3 * (size_t)n_, d_stage_c_, false, &vo));
        export_kernel<T><<<nb, 256, 0, stream_>>>((int)n_, path_ == 0 ? g_ap_ : g_, d_pos4_.as<T4>(), d_vel4_.as<T4>(), d_orig_.as<int>(), cm,
                                                  xo, vo);
        launches_++;
        MB_TRY(view_out_done(coords, xo, 3 * (size_t)n_));
        MB_TRY(view_out_done(vels, vo, 3 * (size_t)n_));
        return finish_call();
    }

    // ------------------------------------------------------------------------------------------
    int remove_cm(void* vels) override {
        MB_TRY(prepare());
        if (!vels) return set_error(MB_ERR_INVALID, "null velocities");
        T* v = nullptr;
        MB_TRY(view_out(vels, 3 * (size_t)n_, d_stage_c_, true, &v));
        double s[3];
        MB_TRY(reduce_to_host(momentum_kernel<T>, v, 3, s));
        subtract_velocity_kernel<T><<<(int)((n_ + 255) / 256), 256, 0, stream_>>>((int)n_, (T)(s[0] / total_mass_), (T)(s[1] / total_mass_),
                                                                                (T)(s[2] / total_mass_), v);
        launches_++;
        MB_TRY(view_out_done(vels, v, 3 * (size_t)n_));
        MB_CUDA(cudaStreamSynchronize(stream_));
        return MB_OK;
    }
    int kinetic_energy(const void* vels, double* out) override {
        MB_TRY(prepare());
        if (!vels || !out) return set_error(MB_ERR_INVALID, "null argument");
        const T* vc = nullptr;
        MB_TRY(view_in(vels, 3 * (size_t)n_, d_stage_c_, &vc));
        return reduce_to_host(kinetic_kernel<T>, vc, 1, out);
    }
    // kinetic energy tensor 1/2 sum m v (x) v (src/energy.jl:56-70) into out9 (3x3, symmetric, host doubles)
    int kinetic_tensor(const void* vels, double* out9) override {
        MB_TRY(prepare());
        if (!vels || !out9) return set_error(MB_ERR_INVALID, "null argument");
        const T* vc = nullptr;
        MB_TRY(view_in(vels, 3 * (size_t)n_, d_stage_c_, &vc));
        double k[6];
        MB_TRY(reduce_to_host(kinetic_tensor_kernel<T>, vc, 6, k));
        out9[0] = k[0]; out9[4] = k[1]; out9[8] = k[2];
        out9[1] = out9[3] = k[3]; out9[2] = out9[6] = k[4]; out9[5] = out9[7] = k[5];
        return MB_OK;
    }
    // random_velocities!(sys, temp; rng) on the device (src/spatial.jl:819-831): fills vels (n x 3, host or device)
    int random_velocities(void* vels, double kT, uint64_t ctr1, uint64_t key) override {
        MB_TRY(prepare());
        if (!vels || !(kT >= 0)) return set_error(MB_ERR_INVALID, "mb_random_velocities: null velocities or negative kT");
        T* vo = nullptr;
        MB_TRY(view_out(vels, 3 * (size_t)n_, d_stage_c_, false, &vo));
        const int nb = (int)((n_ + 255) / 256);
        random_velocities_kernel<T><<<nb, 256, 0, stream_>>>((int)n_, (T)kT, d_mass_in_.as<T>(), (uint32_t)ctr1, (uint32_t)(ctr1 >> 32),
                                                             (uint32_t)key, (uint32_t)(key >> 32), vo);
        launches_++;
        MB_TRY(view_out_done(vels, vo, 3 * (size_t)n_));
        MB_CUDA(cudaStreamSynchronize(stream_));
        return MB_OK;
    }
    int rebuild(const void* coords) override {
        MB_TRY(prepare());
        if (path_ == 0) return MB_OK;
        const T* xc = nullptr;
        MB_TRY(view_in(coords, 3 * (size_t)n_, d_stage_a_, &xc));
        have_list_ = false;
        MB_TRY(sync_state_from(xc, nullptr));
        MB_CUDA(cudaStreamSynchronize(stream_));
        return MB_OK;
    }
    int stats(mb_stats_t* o) override {
        memset(o, 0, sizeof(*o));
        o->n_atoms = n_;
        o->n_force_evals = n_force_evals_;
        o->n_steps = n_steps_;
        o->path = path_;
        o->r_list = r_list_;
        o->kernel_launches = launches_;
        o->graph_mode = graph_used_ ? 1 : (graph_failed_ ? -1 : 0);
        o->reserved_ = dc_.decomposed() ? dc_.auto_every_ : 0;
        o->peer_transport = (dc_.decomposed() && dc_.p2p_active()) ? 1 : 0;
        prof_.collect();
        o->force_ms = prof_.ms[Prof::FORCE]; o->force_launches = prof_.count[Prof::FORCE];
        o->vv_ms = prof_.ms[Prof::VV]; o->vv_launches = prof_.count[Prof::VV];
        o->rebuild_ms = prof_.ms[Prof::REBUILD]; o->rebuild_launches = prof_.count[Prof::REBUILD];
        if (d_ctl_.p && !dirty_) {
            Control c;
            MB_TRY(read_ctl(c));
            o->n_rebuilds = (int64_t)c.n_rebuilds;
            o->n_pairs_in_list = (int64_t)c.n_pairs;
            o->max_neighbors = c.max_neighbors;
            o->max_halo = c.max_halo;
            o->violations = c.violations;
            o->n_prunes = 0;
        }
        if (path_ == 1 && have_list_) {
            o->n_list_entries = (int64_t)n_ * g_.stride;
            o->n_bricks = g_.nbricks;
            for (int d = 0; d < 3; d++) { o->n_cells[d] = g_.nc[d]; o->brick_dims[d] = g_.b[d]; }
            o->halo_capacity = g_.halo_cap;
            o->list_stride = g_.stride;
        }
        return MB_OK;
    }

   private:
    cudaStream_t stream_;
    int sm_count_ = 148;
    size_t smem_optin_ = 232448;
    const EnvSwitches env_;  // read at construction
    int64_t n_ = 0;
    std::vector<T> h_mass_, h_charge_, h_sigma_, h_eps_, h_eps_raw_;
    double box_[3];
    std::vector<mb_inter_t> inters_;
    std::vector<int> ex_ptr_, ex_idx_, sp_ptr_, sp_idx_;
    int max_special_host_ = 0;
    double r_list_ = 0, skin_ = 0, cap_scale_ = 1.0, total_mass_ = 0;
    int rebuild_every_ = 0;
    int user_b_[3] = {0, 0, 0};
    bool dirty_ = true, have_list_ = false;
    int cutm_ = CUTM_PLAIN;  // cutoff family of the kernel variant (pair.cuh)
    int path_ = 0;
    PairParams<T> P_;
    Geom<T> g_, g_ap_;
    Tric<T> tric_ = {};  // TriclinicBoundary (on = 0: cubic / rectangular box)
    int64_t launches_ = 0, n_force_evals_ = 0, n_steps_ = 0, graph_step_launches_ = 0;
    Prof prof_;
    cudaGraph_t graph_ = nullptr;
    cudaGraphExec_t graph_exec_ = nullptr;
    GraphKey graph_key_;
    bool graph_failed_ = false, graph_used_ = false, own_stream_ = false;
    int geom_version_ = 0;
    Decomp<T> dc_;         // multi-GPU state and transport (decomp.cuh)
    BondedHost<T> bonded_; // specific interaction lists (specific.cuh)
    PmeHost<T> pme_;       // PME (pme_host.cuh)
    Dispersion disp_;      // LJDispersionCorrection (specific.cuh)
    DevBuf d_mass_in_, d_charge_in_, d_ljp_in_;
    DevBuf d_pos4_, d_vel4_, d_f4_, d_xref4_, d_lj2_, d_orig_, d_inv_orig_, d_mass_;
    DevBuf d_pos4_t_, d_vel4_t_, d_lj2_t_, d_orig_t_, d_mass_t_;
    DevBuf d_ctl_, d_cm_, d_stage_a_, d_stage_b_, d_stage_c_, d_scalars_;
    DevBuf d_ex_ptr_, d_ex_idx_, d_sp_ptr_, d_sp_idx_;
    DevBuf d_cid_, d_perm_, d_cell_count_, d_cell_start_, d_cell_fill_;
    DevBuf d_hdrs_, d_runs_, d_irows_, d_hcs_, d_counts_, d_list_, d_slist_;
    DevBuf d_erow_total_, d_erow_start_, d_erow_fill_, d_ecell_start_;  // extended (ghost-padded) grid
    DevBuf d_ext_of_, d_gptr_, d_ghosts_, d_pos4e_, d_lj2e_, d_orig_e_;    // slot -> extended map, ghost table, extended arrays
    DevBuf d_task_tab_, d_sched_;  // per-brick task tables; brick ticket + finished-CTA counter of the force kernel
    int force_grid_ = 0;           // CTAs of the last force launch (= number of energy partials)
    DevBuf d_partial_, d_pe_partial_;
};

}  // namespace mb

// ================================================================================================
// C ABI
// ================================================================================================
struct mb_ctx {
    std::unique_ptr<mb::EngineBase> e;
    int device;
    int dtype;
};

#define MB_CTX_GUARD(ctx)                                                         \
    if (!(ctx) || !(ctx)->e) return mb::set_error(MB_ERR_INVALID, "null context"); \
    if (cudaSetDevice((ctx)->device) != cudaSuccess) return mb::set_error(MB_ERR_CUDA, "cudaSetDevice failed")

extern "C" {

const char* mb_last_error(void) { return mb::g_last_error.c_str(); }

int mb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int mb_ctx_create(int device, int dtype, void* cuda_stream, mb_ctx** out) {
    if (!out) return mb::set_error(MB_ERR_INVALID, "out is null");
    *out = nullptr;
    if (dtype != 32 && dtype != 64) return mb::set_error(MB_ERR_INVALID, "dtype must be 32 or 64");
    int n = mb_device_count();
    if (n <= 0) return mb::set_error(MB_ERR_NOGPU, "no CUDA device visible: libmollyb200 has no CPU fallback");
    if (device < 0 || device >= n) return mb::set_error(MB_ERR_INVALID, "device index out of range");
    if (cudaSetDevice(device) != cudaSuccess) return mb::set_error(MB_ERR_CUDA, "cudaSetDevice failed");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return mb::set_error(MB_ERR_CUDA, "cudaGetDeviceProperties failed");
    if (prop.major < 10)
        return mb::set_error(MB_ERR_NOGPU, std::string("device ") + prop.name + " is not sm_100-class; this library is built for sm_100a only");
    mb_ctx* c = new mb_ctx();
    c->device = device;
    c->dtype = dtype;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(cuda_stream);
    if (dtype == 32) c->e.reset(new mb::Engine<float>(device, s));
#ifndef MB_EXP_FAST
    else c->e.reset(new mb::Engine<double>(device, s));
#else
    else { delete c; return mb::set_error(MB_ERR_INVALID, "experiment build: Float32 only"); }
#endif
    *out = c;
    return MB_OK;
}
void mb_ctx_destroy(mb_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    delete ctx;
}
int mb_set_atoms(mb_ctx* ctx, int64_t n, const void* atoms_aos) { MB_CTX_GUARD(ctx); return ctx->e->set_atoms_aos(n, atoms_aos); }
int mb_set_atoms_soa(mb_ctx* ctx, int64_t n, const void* mass, const void* charge, const void* sigma, const void* eps) {
    MB_CTX_GUARD(ctx);
    return ctx->e->set_atoms_soa(n, mass, charge, sigma, eps);
}
int mb_set_box(mb_ctx* ctx, const double side[3]) { MB_CTX_GUARD(ctx); return ctx->e->set_box(side); }
int mb_set_box_triclinic(mb_ctx* ctx, const double basis_vectors[9]) {
    MB_CTX_GUARD(ctx);
    if (!basis_vectors) return mb::set_error(MB_ERR_INVALID, "mb_set_box_triclinic: null basis");
    return ctx->e->set_box_triclinic(basis_vectors);
}
int mb_set_inters(mb_ctx* ctx, int n_inters, const mb_inter_t* inters) { MB_CTX_GUARD(ctx); return ctx->e->set_inters(n_inters, inters); }
int mb_set_exceptions(mb_ctx* ctx, int64_t n_excl, const int32_t* ei, const int32_t* ej, int64_t n_spec, const int32_t* si,
                      const int32_t* sj) {
    MB_CTX_GUARD(ctx);
    return ctx->e->set_exceptions(n_excl, ei, ej, n_spec, si, sj);
}
int mb_set_neighbor_policy(mb_ctx* ctx, double r_list, int rebuild_every) {
    MB_CTX_GUARD(ctx);
    return ctx->e->set_neighbor_policy(r_list, rebuild_every);
}
int mb_forces(mb_ctx* ctx, const void* coords, void* fs_mat, void* virial, int64_t step_n) {
    MB_CTX_GUARD(ctx);
    if (!fs_mat) return mb::set_error(MB_ERR_INVALID, "fs_mat is null");
    return ctx->e->forces_energy(coords, fs_mat, nullptr, virial, step_n, false);
}
int mb_energy(mb_ctx* ctx, const void* coords, void* pe, int64_t step_n) {
    MB_CTX_GUARD(ctx);
    if (!pe) return mb::set_error(MB_ERR_INVALID, "pe is null");
    return ctx->e->forces_energy(coords, nullptr, pe, nullptr, step_n, false);
}
int mb_forces_energy(mb_ctx* ctx, const void* coords, void* fs_mat, void* pe, void* virial, int64_t step_n) {
    MB_CTX_GUARD(ctx);
    return ctx->e->forces_energy(coords, fs_mat, pe, virial, step_n, false);
}
int mb_forces_energy_all(mb_ctx* ctx, const void* coords, void* fs_mat, void* pe, int64_t step_n) {
    MB_CTX_GUARD(ctx);
    return ctx->e->forces_energy(coords, fs_mat, pe, nullptr, step_n, true);
}
int mb_set_specific(mb_ctx* ctx, int kind, int64_t n_terms, const int32_t* atom_idx, const double* params) {
    MB_CTX_GUARD(ctx);
    return ctx->e->set_specific(kind, n_terms, atom_idx, params);
}
int mb_set_pme(mb_ctx* ctx, double r_cut, double error_tol, int order, double eps_r, int64_t n_pairs, const int32_t* pi, const int32_t* pj) {
    MB_CTX_GUARD(ctx);
    return ctx->e->set_pme(r_cut, error_tol, order, eps_r, n_pairs, pi, pj);
}
int mb_set_lj_dispersion_correction(mb_ctx* ctx, double dist_cutoff) { MB_CTX_GUARD(ctx); return ctx->e->set_dispersion(dist_cutoff); }
int mb_random_velocities(mb_ctx* ctx, void* vels, double kT, uint64_t rng_ctr1, uint64_t rng_key) {
    MB_CTX_GUARD(ctx);
    return ctx->e->random_velocities(vels, kT, rng_ctr1, rng_key);
}
int mb_kinetic_energy_tensor(mb_ctx* ctx, const void* vels, double* ke_tensor9_host) { MB_CTX_GUARD(ctx); return ctx->e->kinetic_tensor(vels, ke_tensor9_host); }
int mb_simulate_vv(mb_ctx* ctx, void* coords, void* vels, const mb_vv_params_t* p) { MB_CTX_GUARD(ctx); return ctx->e->simulate_vv(coords, vels, p); }
int mb_remove_cm_motion(mb_ctx* ctx, void* vels) { MB_CTX_GUARD(ctx); return ctx->e->remove_cm(vels); }
int mb_kinetic_energy(mb_ctx* ctx, const void* vels, double* ke_host) { MB_CTX_GUARD(ctx); return ctx->e->kinetic_energy(vels, ke_host); }
int mb_rebuild_neighbors(mb_ctx* ctx, const void* coords) { MB_CTX_GUARD(ctx); return ctx->e->rebuild(coords); }
int mb_stats(mb_ctx* ctx, mb_stats_t* host_out) {
    MB_CTX_GUARD(ctx);
    if (!host_out) return mb::set_error(MB_ERR_INVALID, "null stats");
    return ctx->e->stats(host_out);
}
int mb_synchronize(mb_ctx* ctx) { MB_CTX_GUARD(ctx); return ctx->e->synchronize(); }
int mb_set_capacity_scale(mb_ctx* ctx, double scale) { MB_CTX_GUARD(ctx); return ctx->e->set_capacity_scale(scale); }
int mb_set_launch_config(mb_ctx* ctx, const int32_t brick_dims[3], int32_t lanes_per_atom) {
    MB_CTX_GUARD(ctx);
    return ctx->e->set_launch_config(brick_dims, lanes_per_atom);
}
int mb_set_profiling(mb_ctx* ctx, int enable) { MB_CTX_GUARD(ctx); return ctx->e->set_profiling(enable); }
int mb_comm_unique_id(void* out128) {
    if (!out128) return mb::set_error(MB_ERR_INVALID, "null output");
    if (!mb::g_nccl.load()) return mb::set_error(MB_ERR_INVALID, "libnccl.so.2 could not be loaded");
    mb::ncclUniqueId id;
    if (mb::g_nccl.GetUniqueId(&id) != mb::ncclSuccess) return mb::set_error(MB_ERR_CUDA, "ncclGetUniqueId failed");
    memcpy(out128, &id, sizeof(id));
    return MB_OK;
}
int mb_decomp_plan(int ncz, int halo_layers, int nranks, int rank, const int32_t* layer_start, int32_t* send_out, int32_t* n_send,
                   int32_t* recv_out, int32_t* n_recv, int capacity) {
    if (ncz < 1 || nranks < 1 || nranks > ncz || rank < 0 || rank >= nranks || !layer_start || !send_out || !recv_out || !n_send || !n_recv)
        return mb::set_error(MB_ERR_INVALID, "mb_decomp_plan: bad arguments");
    std::vector<mb::DecompSeg> snd, rcv;
    mb::decomp_plan(ncz, halo_layers, nranks, rank, layer_start, snd, rcv);
    if ((int)snd.size() > capacity || (int)rcv.size() > capacity) return mb::set_error(MB_ERR_CAPACITY, "mb_decomp_plan: capacity");
    for (size_t k = 0; k < snd.size(); k++) { send_out[3 * k] = snd[k].peer; send_out[3 * k + 1] = snd[k].start; send_out[3 * k + 2] = snd[k].count; }
    for (size_t k = 0; k < rcv.size(); k++) { recv_out[3 * k] = rcv[k].peer; recv_out[3 * k + 1] = rcv[k].start; recv_out[3 * k + 2] = rcv[k].count; }
    *n_send = (int32_t)snd.size();
    *n_recv = (int32_t)rcv.size();
    return MB_OK;
}
int mb_pme_plan(const double box[3], double r_cut, double error_tol, int order, double* alpha_out, int32_t mesh_out[3],
                double* moduli_out, int capacity) {
    if (!box || !alpha_out || !mesh_out || !(r_cut > 0) || !(error_tol > 0 && error_tol < 0.5) || order < 3 || order > 8)
        return mb::set_error(MB_ERR_INVALID, "mb_pme_plan: bad arguments");
    std::vector<double> moduli[3];
    int K[3];
    mb::pme_plan_host(box, r_cut, error_tol, order, alpha_out, K, moduli);
    for (int d = 0; d < 3; d++) mesh_out[d] = K[d];
    if (moduli_out) {
        if (K[0] + K[1] + K[2] > capacity) return mb::set_error(MB_ERR_CAPACITY, "mb_pme_plan: capacity");
        size_t o = 0;
        for (int d = 0; d < 3; d++)
            for (double v : moduli[d]) moduli_out[o++] = v;
    }
    return MB_OK;
}
int mb_comm_init(mb_ctx* ctx, const void* unique_id128, int rank, int nranks) {
    MB_CTX_GUARD(ctx);
    return ctx->e->comm_init(unique_id128, rank, nranks);
}

}  // extern "C"
