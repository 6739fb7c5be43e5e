// decomp.cuh — host side of the multi-GPU run (DESIGN.md §5): the slab decomposition plan and Decomp<T>, which owns
// every piece of multi-GPU state of an engine: the NCCL communicator, rank ownership of bricks and slots, the halo
// segments, the adaptive rebuild interval and the NVLink peer-memory transport (peer.cuh). The engine hands it the
// geometry and device arrays it needs as arguments; kernels are launched on the engine's stream.
#pragma once
#include <algorithm>
#include <cmath>

#include "dynlib.h"
#include "host_util.h"
#include "vv.cuh"

namespace mb {

// ---------------------------------------------------------------------------------------------
// Slab decomposition plan (pure host logic, exported as mb_decomp_plan so it can be tested without a GPU):
// rank q owns cell layers [q*ncz/P, (q+1)*ncz/P); it needs the h layers below and above its slab (periodic).
// Segments are contiguous slot ranges [start, start+count) taken from layer_start (ncz + 1 prefix offsets).
// Both ends enumerate the segments of a (sender, receiver) pair in the receiver's order, so the grouped
// ncclSend/ncclRecv calls match up.
// ---------------------------------------------------------------------------------------------
struct DecompSeg { int peer, start, count; };
static inline int decomp_layer_lo(int q, int ncz, int nranks) { return (int)(((long long)q * ncz) / nranks); }
static inline int decomp_layer_owner(int layer, int ncz, int nranks) {
    for (int q = 0; q < nranks; q++)
        if (layer >= decomp_layer_lo(q, ncz, nranks) && layer < decomp_layer_lo(q + 1, ncz, nranks)) return q;
    return nranks - 1;
}
static void decomp_needed(int q, int ncz, int h, int nranks, std::vector<int>& out) {
    out.clear();
    const int lo = decomp_layer_lo(q, ncz, nranks), hi = decomp_layer_lo(q + 1, ncz, nranks);
    std::vector<char> seen(ncz, 0);
    for (int l = lo; l < hi; l++) seen[l] = 1;
    for (int l = lo - h; l < lo; l++) { int w = ((l % ncz) + ncz) % ncz; if (!seen[w]) { seen[w] = 1; out.push_back(w); } }
    for (int l = hi; l < hi + h; l++) { int w = l % ncz; if (!seen[w]) { seen[w] = 1; out.push_back(w); } }
}
static void decomp_plan(int ncz, int h, int nranks, int rank, const int* layer_start, std::vector<DecompSeg>& send,
                        std::vector<DecompSeg>& recv) {
    auto add = [&](std::vector<DecompSeg>& v, int peer, int layer) {
        int st = layer_start[layer], cnt = layer_start[layer + 1] - st;
        if (!v.empty() && v.back().peer == peer && v.back().start + v.back().count == st) v.back().count += cnt;
        else v.push_back({peer, st, cnt});
    };
    send.clear();
    recv.clear();
    std::vector<int> need;
    decomp_needed(rank, ncz, h, nranks, need);
    for (int l : need) add(recv, decomp_layer_owner(l, ncz, nranks), l);
    for (int q = 0; q < nranks; q++) {
        if (q == rank) continue;
        decomp_needed(q, ncz, h, nranks, need);
        for (int l : need)
            if (decomp_layer_owner(l, ncz, nranks) == rank) add(send, q, l);
    }
}

// spatial decomposition (z-slabs of cell layers; one rank per GPU)
template <typename T>
struct Decomp {
    using T4 = typename VT<T>::T4;

    cudaStream_t stream_ = nullptr;      // the engine's stream
    ncclComm_t comm_ = nullptr;
    int rank_ = 0, nranks_ = 1;
    int own_b0_ = 0, own_nb_ = 0;        // this rank's bricks (static for a geometry)
    bool own_valid_ = false;             // ownership derived from the current sort
    int since_rebuild_ = 0;              // MD steps since the last rebuild of a decomposed run (host count, same on every rank)
    int adapt_span_ = 0;                 // longest such count within the current call
    int build_b0_ = 0, build_nb_ = -1;   // brick range the list builder covers (-1 = all)
    int own_s0_ = 0, own_n_ = 0;         // this rank's slots (changes at every rebuild)
    int auto_every_ = 20;                // rebuild interval of decomposed runs when the policy is displacement-triggered
    std::vector<int> layer_start_;       // slot index of the first atom of every cell layer (ncz + 1)
    std::vector<DecompSeg> halo_send_, halo_recv_;
    DevBuf d_layer_start_, d_mom_;
    // peer-memory transport (peer.cuh): IPC-mapped position arrays and PeerComm blocks of the other ranks
    bool p2p_ = false;
    void* p2p_pos_base_ = nullptr;            // the extended position allocation the peers have mapped
    DevBuf d_comm_, d_ipc_;
    std::vector<void*> peer_pos_, peer_comm_; // [rank]; own entries point at the local buffers
    unsigned long long epoch_ = 0;            // force evaluations of decomposed runs (same on every rank)
    bool plan_fits_ = false;
    PeerWait gate_ = {};                      // one-shot gate of the next force launch, set by the decomposed step
    unsigned long long cm_deferred_epoch_ = 0;
    int plan_key_[3] = {-1, -1, -1};

    bool decomposed() const { return nranks_ > 1; }
    double* mom() const { return d_mom_.as<double>(); }  // [0,3) this slab's sum(m v), [4,7) the global one
    int own_brick0() const { return build_nb_ < 0 ? 0 : build_b0_; }
    int own_nbricks(int nbricks) const { return build_nb_ < 0 ? nbricks : build_nb_; }
    int layer_lo(int q, const Geom<T>& g) const { return decomp_layer_lo(q, g.nc[2], nranks_); }
    // slot ranges and halo segments follow from the cell layer offsets of the current sort (host copy)
    int interval(int rebuild_every) const { return rebuild_every > 0 ? rebuild_every : auto_every_; }
    int update_ownership(const Geom<T>& g, const int* d_cell_start) {
        own_valid_ = true;
        const int ncz = g.nc[2], per_layer = g.nc[0] * g.nc[1];
        layer_start_.resize(ncz + 1);
        MB_CUDA(d_layer_start_.ensure((size_t)(ncz + 1) * sizeof(int)));
        MB_CUDA(cudaMemcpy2DAsync(d_layer_start_.p, sizeof(int), d_cell_start, (size_t)per_layer * sizeof(int), sizeof(int),
                                  (size_t)ncz + 1, cudaMemcpyDeviceToDevice, stream_));
        MB_CUDA(cudaMemcpyAsync(layer_start_.data(), d_layer_start_.p, (size_t)(ncz + 1) * sizeof(int), cudaMemcpyDeviceToHost, stream_));
        MB_CUDA(cudaStreamSynchronize(stream_));
        const int nbxy = g.nb[0] * g.nb[1];
        own_b0_ = layer_lo(rank_, g) * nbxy;
        own_nb_ = (layer_lo(rank_ + 1, g) - layer_lo(rank_, g)) * nbxy;
        own_s0_ = layer_start_[layer_lo(rank_, g)];
        own_n_ = layer_start_[layer_lo(rank_ + 1, g)] - own_s0_;
        decomp_plan(ncz, g.h, nranks_, rank_, layer_start_.data(), halo_send_, halo_recv_);
        // The peer-memory transport carries at most MB_MAX_SEG segments / peers per rank. Whether the plan fits must be
        // the same answer on every rank and every step, so it is evaluated for all ranks on unit-sized layers
        // (the segment structure depends only on ncz, h and the rank count).
        if (plan_key_[0] != ncz || plan_key_[1] != g.h || plan_key_[2] != nranks_) {
            plan_key_[0] = ncz; plan_key_[1] = g.h; plan_key_[2] = nranks_;
            std::vector<int> unit(ncz + 1);
            for (int l = 0; l <= ncz; l++) unit[l] = l;
            plan_fits_ = nranks_ <= MB_MAX_RANKS;
            std::vector<DecompSeg> sd, rv;
            std::vector<int> a, b;
            for (int q = 0; q < nranks_ && plan_fits_; q++) {
                decomp_plan(ncz, g.h, nranks_, q, unit.data(), sd, rv);
                distinct_peers(sd, a);
                distinct_peers(rv, b);
                if ((int)sd.size() > MB_MAX_SEG || (int)a.size() > MB_MAX_SEG || (int)b.size() > MB_MAX_SEG) plan_fits_ = false;
            }
        }
        return MB_OK;
    }
    bool p2p_active() const { return p2p_ && plan_fits_; }
    // Decomposed runs rebuild at a fixed interval (every rank must take the same branch without a host round trip).
    // The interval for the NEXT call is derived from the largest displacement any interval of this call reached:
    // n_next = 0.8 * n * (skin/2) / d_max, agreed between ranks with one max-all-reduce. Violations are still counted.
    int adapt_interval(const Control* ctl, double skin, int64_t& launches) {
        // largest displacement any rebuild interval of this call reached (device) -> max over ranks -> host; the only host
        // wait is the one the end of the call has anyway
        float* dbuf = reinterpret_cast<float*>(d_mom_.as<double>() + 7);
        max_disp_kernel<<<1, 1, 0, stream_>>>(ctl, dbuf);
        launches++;
        MB_NCCL(g_nccl.AllReduce(dbuf, dbuf, 1, (ncclDataType_t)7 /* ncclFloat32 */, (ncclRedOp_t)2 /* ncclMax */, comm_, stream_));
        float d2 = 0.f;
        MB_CUDA(cudaMemcpyAsync(&d2, dbuf, sizeof(float), cudaMemcpyDeviceToHost, stream_));
        MB_CUDA(cudaStreamSynchronize(stream_));
        if (d2 > 0.f && skin > 0) {
            // d2 was reached within adapt_span_ steps of a rebuild; displacements grow at most linearly in time
            double n_next = 0.8 * std::max(adapt_span_, 1) * (0.5 * skin) / std::sqrt((double)d2);
            auto_every_ = (int)std::min(400.0, std::max(5.0, std::floor(n_next)));
        }
        return MB_OK;
    }
    // forward halo exchange of positions (x, y, z, q as 16/32-byte records): grouped NCCL send/recv between slabs; the
    // caller refreshes the extended array for the received segments
    int halo_exchange(T4* pos4) {
        MB_NCCL(g_nccl.GroupStart());
        for (auto& sg : halo_send_)
            if (sg.count > 0) MB_NCCL(g_nccl.Send(pos4 + sg.start, (size_t)sg.count * sizeof(T4), ncclChar, sg.peer, comm_, stream_));
        for (auto& sg : halo_recv_)
            if (sg.count > 0) MB_NCCL(g_nccl.Recv(pos4 + sg.start, (size_t)sg.count * sizeof(T4), ncclChar, sg.peer, comm_, stream_));
        MB_NCCL(g_nccl.GroupEnd());
        return MB_OK;
    }
    // replicate the owned segments of positions and velocities on every rank (rebuild / export)
    int allgather_state(const Geom<T>& g, T4* pos4, T4* vel4) {
        MB_NCCL(g_nccl.GroupStart());
        for (int q = 0; q < nranks_; q++) {
            const int st = layer_start_[layer_lo(q, g)], cnt = layer_start_[layer_lo(q + 1, g)] - st;
            if (cnt <= 0) continue;
            MB_NCCL(g_nccl.Broadcast(pos4 + st, pos4 + st, (size_t)cnt * sizeof(T4), ncclChar, q, comm_, stream_));
            MB_NCCL(g_nccl.Broadcast(vel4 + st, vel4 + st, (size_t)cnt * sizeof(T4), ncclChar, q, comm_, stream_));
        }
        MB_NCCL(g_nccl.GroupEnd());
        return MB_OK;
    }
    // ---- peer-memory transport (peer.cuh) -------------------------------------------------------------------
    void p2p_close() {
        for (int r = 0; r < (int)peer_pos_.size(); r++) {
            if (r == rank_) continue;
            if (peer_pos_[r]) cudaIpcCloseMemHandle(peer_pos_[r]);
            if (peer_comm_[r]) cudaIpcCloseMemHandle(peer_comm_[r]);
        }
        peer_pos_.clear();
        peer_comm_.clear();
        p2p_ = false;
        p2p_pos_base_ = nullptr;
    }
    // Collective: every rank exports its (extended) position array and its PeerComm block as CUDA IPC handles, the handles
    // travel by one ncclAllGather, and every rank maps the others'. Any failure on any rank (no peer access, IPC not
    // permitted in this container, too many ranks, allow = false) leaves ALL ranks on the NCCL transport.
    int p2p_setup(void* pos4e, bool allow) {
        if (p2p_pos_base_ == pos4e && !peer_pos_.empty()) return MB_OK;  // mapping is current
        p2p_close();
        p2p_pos_base_ = pos4e;
        peer_pos_.assign(nranks_, nullptr);
        peer_comm_.assign(nranks_, nullptr);
        int ok = allow && nranks_ <= MB_MAX_RANKS;
        struct Rec { cudaIpcMemHandle_t pos, comm; };
        static_assert(sizeof(Rec) == 128, "two 64-byte IPC handles");
        // 2 MiB so the block is an allocation of its own; zeroed before any peer can learn its address
        MB_CUDA(d_comm_.ensure(2u << 20));
        MB_CUDA(cudaMemsetAsync(d_comm_.p, 0, sizeof(PeerComm), stream_));
        const unsigned long long magic = 0x6d62323030ull + (unsigned long long)rank_;
        MB_CUDA(cudaMemcpyAsync(reinterpret_cast<char*>(d_comm_.p) + offsetof(PeerComm, magic), &magic, sizeof(magic),
                                cudaMemcpyHostToDevice, stream_));
        Rec mine;
        memset(&mine, 0, sizeof(mine));
        if (ok && cudaIpcGetMemHandle(&mine.pos, pos4e) != cudaSuccess) { ok = 0; cudaGetLastError(); }
        if (ok && cudaIpcGetMemHandle(&mine.comm, d_comm_.p) != cudaSuccess) { ok = 0; cudaGetLastError(); }
        MB_CUDA(d_ipc_.ensure((size_t)(nranks_ + 1) * sizeof(Rec) + 16));
        Rec* d_all = d_ipc_.as<Rec>();
        MB_CUDA(cudaMemcpyAsync(d_all + nranks_, &mine, sizeof(Rec), cudaMemcpyHostToDevice, stream_));
        MB_NCCL(g_nccl.AllGather(d_all + nranks_, d_all, sizeof(Rec), ncclChar, comm_, stream_));
        std::vector<Rec> all(nranks_);
        MB_CUDA(cudaMemcpyAsync(all.data(), d_all, (size_t)nranks_ * sizeof(Rec), cudaMemcpyDeviceToHost, stream_));
        MB_CUDA(cudaStreamSynchronize(stream_));
        for (int r = 0; r < nranks_ && ok; r++) {
            if (r == rank_) { peer_pos_[r] = pos4e; peer_comm_[r] = d_comm_.p; continue; }
            if (cudaIpcOpenMemHandle(&peer_pos_[r], all[r].pos, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
                cudaIpcOpenMemHandle(&peer_comm_[r], all[r].comm, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                ok = 0;
                cudaGetLastError();
                break;
            }
            unsigned long long got = 0;  // the mapping must show the owner's tag
            if (cudaMemcpy(&got, reinterpret_cast<char*>(peer_comm_[r]) + offsetof(PeerComm, magic), sizeof(got),
                           cudaMemcpyDeviceToHost) != cudaSuccess || got != 0x6d62323030ull + (unsigned long long)r) {
                ok = 0;
                cudaGetLastError();
            }
        }
        // agree: min over ranks
        float okf = (float)ok;
        float* dbuf = reinterpret_cast<float*>(reinterpret_cast<char*>(d_ipc_.p) + (size_t)(nranks_ + 1) * sizeof(Rec));
        MB_CUDA(cudaMemcpyAsync(dbuf, &okf, sizeof(float), cudaMemcpyHostToDevice, stream_));
        MB_NCCL(g_nccl.AllReduce(dbuf, dbuf, 1, (ncclDataType_t)7 /* ncclFloat32 */, (ncclRedOp_t)3 /* ncclMin */, comm_, stream_));
        MB_CUDA(cudaMemcpyAsync(&okf, dbuf, sizeof(float), cudaMemcpyDeviceToHost, stream_));
        MB_CUDA(cudaStreamSynchronize(stream_));
        if (okf < 0.5f) {
            void* keep = p2p_pos_base_;
            p2p_close();
            p2p_pos_base_ = keep;            // do not retry on every call
            peer_pos_.assign(nranks_, nullptr);
            return MB_OK;
        }
        p2p_ = true;
        return MB_OK;
    }
    PeerComm* comm_of(int r) const { return reinterpret_cast<PeerComm*>(peer_comm_[r]); }
    // distinct peers of a segment list, in first-appearance order
    static void distinct_peers(const std::vector<DecompSeg>& v, std::vector<int>& out) {
        out.clear();
        for (auto& sg : v)
            if (sg.count > 0 && std::find(out.begin(), out.end(), sg.peer) == out.end()) out.push_back(sg.peer);
    }
    PeerPush<T> make_push(unsigned long long epoch, bool with_data) const {
        PeerPush<T> ps;
        memset(&ps, 0, sizeof(ps));
        ps.epoch = epoch;
        std::vector<int> peers;
        distinct_peers(halo_send_, peers);
        if (with_data)
            for (auto& sg : halo_send_) {
                if (sg.count <= 0) continue;
                ps.start[ps.n_seg] = sg.start;
                ps.count[ps.n_seg] = sg.count;
                ps.dst[ps.n_seg] = reinterpret_cast<T4*>(peer_pos_[sg.peer]);
                ps.n_seg++;
            }
        for (int q : peers) {
            ps.wait_flag[ps.n_peer] = &comm_of(rank_)->read_epoch[q];
            ps.signal_flag[ps.n_peer] = &comm_of(q)->halo_epoch[rank_];
            ps.n_peer++;
        }
        return ps;
    }
    PeerWait make_wait(unsigned long long epoch) const {
        PeerWait w;
        memset(&w, 0, sizeof(w));
        w.epoch = epoch;
        std::vector<int> peers;
        distinct_peers(halo_recv_, peers);
        for (int q : peers) w.flag[w.n++] = &comm_of(rank_)->halo_epoch[q];
        return w;
    }
    PeerSignal make_signal(unsigned long long epoch, bool with_mom) const {
        PeerSignal sg;
        memset(&sg, 0, sizeof(sg));
        sg.epoch = epoch;
        std::vector<int> peers;
        distinct_peers(halo_recv_, peers);
        for (int q : peers) sg.read_flag[sg.n_peer++] = &comm_of(q)->read_epoch[rank_];
        if (with_mom) {
            const int par = (int)(epoch & 1ull);
            sg.n_mom = nranks_;
            for (int r = 0; r < nranks_; r++) {
                sg.mom_dst[r] = comm_of(r)->mom[par][rank_];
                sg.mom_flag[r] = &comm_of(r)->mom_epoch[par][rank_];
            }
        }
        return sg;
    }

    int comm_init(const void* uid, int rank, int nranks) {
        if (nranks < 1 || rank < 0 || rank >= nranks || !uid) return set_error(MB_ERR_INVALID, "mb_comm_init: bad arguments");
        if (!g_nccl.load()) return set_error(MB_ERR_INVALID, "mb_comm_init: libnccl.so.2 could not be loaded");
        p2p_close();
        if (comm_) { g_nccl.CommDestroy(comm_); comm_ = nullptr; }
        rank_ = rank;
        nranks_ = nranks;
        if (nranks > 1) {
            ncclUniqueId id;
            memcpy(&id, uid, sizeof(id));
            MB_NCCL(g_nccl.CommInitRank(&comm_, nranks, id, rank));
            MB_CUDA(d_mom_.ensure(8 * sizeof(double)));
        }
        return MB_OK;
    }
};

}  // namespace mb
