// peer.cuh — NVLink peer-memory transport of the decomposed MD step (SURVEY.md §8(e)).
//
// Every rank holds the whole position array in the SAME slot order (the cell sort is replicated), so a halo
// exchange is "write my boundary slots into the neighbour's array at the same indices". The drift kernel (K1) does
// exactly that with plain stores through IPC-mapped peer pointers while it integrates, and its last CTA publishes
// an epoch flag in the neighbour's PeerComm block; the neighbour's force kernel is gated by a one-warp wait on that
// flag. The per-step sum(m v) for remove_CM_motion! is an all-to-all of 24 bytes written by K2's last CTA and summed
// in rank order (deterministic, identical on every rank). No NCCL call and no host round trip is left in a
// non-rebuild step; NCCL stays for bootstrap, the all-gather at neighbour rebuilds and the export.
//
// Protocol (epoch e = running count of force evaluations, the same number on every rank):
//   K1(e)    waits  read_epoch[p] >= e-1  for every peer p it pushes to (p has finished reading my step e-1 data),
//            stores the new positions locally and into the peers, then sets  peer.halo_epoch[me] = e.
//   wait(e)  spins until halo_epoch[q] >= e for every peer q that pushes to me.
//   force(e), K2(e): K2's last CTA sets  peer.read_epoch[me] = e  for every q that pushes to me, and (CM removal)
//            writes sum(m v) into every rank's mom[e&1][me] followed by mom_epoch[e&1][me] = e.
//   cm(e)    spins until mom_epoch[e&1][r] >= e for all r, adds the nranks partial sums in rank order: done by every
//            CTA of K1(e+1) itself between two steps, by peer_cm_kernel when something else consumes v_cm next.
//   The force kernel's CTAs do wait(e) themselves (ForceOut::gate), so a non-rebuild step is K1 -> force -> K2.
// All waits are bounded (a few seconds of %globaltimer) and trap instead of hanging the GPU.
#pragma once
#include "common.cuh"

namespace mb {

constexpr int MB_MAX_RANKS = 16;
constexpr int MB_MAX_SEG = 8;

struct PeerComm {
    unsigned long long halo_epoch[MB_MAX_RANKS];    // [src]: src's pushes for this epoch have landed in my pos4
    unsigned long long read_epoch[MB_MAX_RANKS];    // [src]: src has finished reading the halo data of this epoch
    unsigned long long mom_epoch[2][MB_MAX_RANKS];  // [parity][src]
    double mom[2][MB_MAX_RANKS][4];                 // [parity][src]: sum(m v) of src's slab
    unsigned long long magic;                       // mapping self-check
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// bounded spin: a peer that never arrives turns into a CUDA error on this rank instead of a hung GPU
__device__ __forceinline__ void spin_until(const unsigned long long* flag, unsigned long long need) {
    if (ld_acquire_sys(flag) >= need) return;
    const unsigned long long t0 = global_timer_ns();
    while (ld_acquire_sys(flag) < need) {
        __nanosleep(64);
        if (global_timer_ns() - t0 > 8000000000ull) __trap();
    }
}

// K1 argument: which owned slot ranges are mirrored into which peer arrays, and the flags around it
template <typename T>
struct PeerPush {
    int n_seg;
    int start[MB_MAX_SEG], count[MB_MAX_SEG];
    typename VT<T>::T4* dst[MB_MAX_SEG];  // peer's extended position array pos4e (same indexing: the cell sort is replicated)
    int n_peer;
    const unsigned long long* wait_flag[MB_MAX_SEG];  // my comm->read_epoch[peer]
    unsigned long long* signal_flag[MB_MAX_SEG];      // peer comm->halo_epoch[me]
    unsigned long long epoch;                          // waits need epoch-1, signals write epoch
    // v_cm of the previous step straight from the momentum all-to-all (replaces peer_cm_kernel between two steps)
    const PeerComm* cm_comm;
    int cm_nranks;                                     // 0: take v_cm from CmState as usual
    unsigned long long cm_epoch;
    double cm_inv_mass;
};

// K2 argument: read-done signals and the momentum all-to-all
struct PeerSignal {
    int n_peer;
    unsigned long long* read_flag[MB_MAX_SEG];  // peer comm->read_epoch[me]
    int n_mom;                                  // 0 or nranks
    double* mom_dst[MB_MAX_RANKS];              // rank r's comm->mom[parity][me]
    unsigned long long* mom_flag[MB_MAX_RANKS]; // rank r's comm->mom_epoch[parity][me]
    unsigned long long epoch;
};

struct PeerWait {
    int n;
    const unsigned long long* flag[MB_MAX_RANKS];
    unsigned long long epoch;
};

// stand-alone signal (after the force evaluation that precedes the first step of a call)
__global__ void peer_signal_kernel(PeerSignal s) {
    if ((int)threadIdx.x < s.n_peer) {
        __threadfence_system();
        st_release_sys(s.read_flag[threadIdx.x], s.epoch);
    }
}

}  // namespace mb
