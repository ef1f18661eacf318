// The multi-GPU combine step over NVLink / NVSwitch peer memory (SURVEY.md section 8e) -- instead of an NCCL all-reduce.
//
// One process per GPU.  Every engine owns a MAILBOX in device memory (cudaMalloc + CUDA IPC handle, mapped by every
// peer): one inbox slot per rank plus control words.  A slot holds the accumulator store in a self-validating form: every
// double travels as two 8-byte words {low half | flag}, {high half | flag} with flag = the epoch number, so the receiver
// knows an element has arrived by looking at the element itself (8-byte stores are single-copy atomic) -- no fence, no
// arrival counter, no remote read-modify-write on the critical path.  After a rank's exhaustive launch
//   non-root:  p2p_push_kernel  writes its store into ITS slot of the root's mailbox (16-byte posted stores over NVLink:
//              172 KB for the 150-SNP locus) and is done;
//   root:      p2p_merge_kernel polls the peers' slots element by element until they carry this epoch's flag, adds them to
//              its store (p2p_gather), and posts `consumed = epoch` into every peer's control word (p2p_root_done; flow
//              control: a peer may only overwrite its slot for epoch k once the root has consumed epoch k-1; peers poll their
//              LOCAL word).  finalize_merge_kernel (engine.cu) does the same inside the finalize.
// Both are ordinary stream-ordered launches: no host synchronisation, no collective library; the epoch counters live in
// device memory so the launches have no per-step argument and replay from a CUDA graph.  Spins are bounded (about a
// minute of clock64) and raise ERR_P2P_TIMEOUT instead of hanging the device.  (Measured alternatives on B200 x 2, 86 KB
// store: system-scope fp64 atomics of the non-zero bins + fence + arrival counter 21-25 us per push; dense stores +
// fence + arrival counter 19 us; NCCL all-reduce 31 us.)
#pragma once
#include "common.cuh"

namespace pipsort {

typedef unsigned long long u64;

constexpr int P2P_MAX_WORLD = 16;
constexpr long long P2P_SPIN_CYCLES = 120000000000ll;   // ~60 s at 1.9 GHz: ranks may reach the combine step far apart

struct P2PPeers {
    u64* ctrl[P2P_MAX_WORLD];   // every rank's control words: [0] arrivals (root's is used), [1] consumed, [2] epoch (local)
    int world, root;
};

__device__ inline bool p2p_spin_ge(const volatile u64* p, u64 target) {
    const long long t0 = clock64();
    while (*p < target) {
        if (clock64() - t0 > P2P_SPIN_CYCLES) return false;
        __nanosleep(64);
    }
    return true;
}

// The mailbox word: a double v as {low half of v | flag}, {high half of v | flag}, flag = the low 32 bits of the epoch.
__device__ __forceinline__ ulonglong2 p2p_encode(double v, u64 flag) {
    const u64 b = (u64)__double_as_longlong(v), f = flag << 32;
    return make_ulonglong2((b & 0xffffffffull) | f, (b >> 32) | f);
}
__device__ __forceinline__ bool p2p_arrived(const ulonglong2& w, u64 flag) { return (w.x >> 32) == flag && (w.y >> 32) == flag; }
__device__ __forceinline__ double p2p_decode(const ulonglong2& w) {
    return __longlong_as_double((long long)((w.x & 0xffffffffull) | (w.y << 32)));
}
__device__ __forceinline__ ulonglong2 p2p_load(const ulonglong2* src) {   // both words in one 16-byte load, past the caches
    ulonglong2 w;
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(w.x), "=l"(w.y) : "l"(src));
    return w;
}

// one element of a peer's slot: spins until both words carry this epoch's flag (8-byte stores are single-copy atomic)
__device__ __forceinline__ double p2p_take(const ulonglong2* src, u64 flag, bool& ok) {
    ulonglong2 w;
    const long long t0 = clock64();
    for (;;) {
        w = p2p_load(src);
        if (p2p_arrived(w, flag)) break;
        if (clock64() - t0 > P2P_SPIN_CYCLES) { ok = false; break; }
        __nanosleep(32);
    }
    return p2p_decode(w);
}

// Element i of the store summed over the GPUs: v (the root's own value) first, then every peer's copy in ascending rank
// (slots: the root's own mailbox, world slots of slot_stride 16-byte elements each; slot r is written by rank r).  Up to 8
// ranks, all peers' copies are requested at once (one round trip, not one per peer: with 7 peers the serial polls were
// most of the step at N = 8) and re-requested until each carries this epoch's flag; beyond that, one peer after the other.
__device__ __forceinline__ double p2p_gather(double v, const ulonglong2* slots, size_t slot_stride, size_t i, const P2PPeers& peers,
                                             int my_rank, u64 flag, bool& ok) {
    if (peers.world <= 8) {
        ulonglong2 wr[8];
        unsigned pend = 0;
#pragma unroll
        for (int r = 0; r < 8; r++)
            if (r < peers.world && r != my_rank) {
                wr[r] = p2p_load(slots + (size_t)r * slot_stride + i);
                pend |= 1u << r;
            }
        const long long t0 = clock64();
        for (;;) {
#pragma unroll
            for (int r = 0; r < 8; r++)
                if ((pend >> r & 1) && p2p_arrived(wr[r], flag)) pend &= ~(1u << r);
            if (!pend) break;
            if (clock64() - t0 > P2P_SPIN_CYCLES) { ok = false; break; }
            __nanosleep(32);
#pragma unroll
            for (int r = 0; r < 8; r++)
                if (pend >> r & 1) wr[r] = p2p_load(slots + (size_t)r * slot_stride + i);
        }
#pragma unroll
        for (int r = 0; r < 8; r++)
            if (r < peers.world && r != my_rank) v += p2p_decode(wr[r]);
        return v;
    }
    for (int r = 0; r < peers.world; r++)
        if (r != my_rank) v += p2p_take(slots + (size_t)r * slot_stride + i, flag, ok);
    return v;
}

// The root's end of a combine kernel, reached by every thread of every block: records a timeout, and the last block to
// finish (every block has then read the slots: the peers may overwrite them) moves this rank to the next epoch and posts
// `consumed = epoch` into every peer's control word.
__device__ __forceinline__ void p2p_root_done(bool ok, u64 epoch, u64* my_ctrl, const P2PPeers& peers, int my_rank, unsigned* done,
                                              double* err_flag) {
    if (!ok) atomicAdd(err_flag, 1.0);
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned d = atomicAdd(done, 1u);
        if (d == gridDim.x - 1) {
            *done = 0;
            my_ctrl[2] = epoch;
            __threadfence_system();
            for (int r = 0; r < peers.world; r++)
                if (r != my_rank) *(volatile u64*)(peers.ctrl[r] + 1) = epoch;   // posted store, nobody waits for it here
        }
    }
}

__global__ void __launch_bounds__(256)
p2p_push_kernel(double* __restrict__ store, size_t n, ulonglong2* __restrict__ my_slot_at_root, u64* __restrict__ my_ctrl,
                unsigned* __restrict__ done, double* __restrict__ err_flag, int clear) {
    __shared__ int ok;
    __shared__ u64 epoch_s;
    // (launched with programmatic stream serialization: resident early, but the store is final only when the kernel
    // before this one in the stream has completed)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // the epoch lives in device memory (control word 2, bumped by the last block) so that the launch has no per-step
    // argument and can be replayed from a CUDA graph
    if (threadIdx.x == 0) {
        epoch_s = *(volatile u64*)(my_ctrl + 2) + 1;
        ok = p2p_spin_ge(my_ctrl + 1, epoch_s - 1) ? 1 : 0;        // the root has consumed the previous epoch's slot
    }
    __syncthreads();
    const u64 flag = epoch_s & 0xffffffffull;
    if (ok) {
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
            const double v = store[i];
            my_slot_at_root[i] = p2p_encode(v, flag);
            if (clear && __double_as_longlong(v)) store[i] = 0.0;   // what has been sent is gone: the push doubles as this rank's reset
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (!ok) atomicAdd(err_flag, 1.0);
        const unsigned d = atomicAdd(done, 1u);
        if (d == gridDim.x - 1) { *done = 0; my_ctrl[2] = epoch_s; }   // local bookkeeping only: next epoch
    }
}

// slots: as p2p_gather takes them
__global__ void __launch_bounds__(256)
p2p_merge_kernel(double* __restrict__ store, const ulonglong2* slots, size_t n, size_t slot_stride, u64* __restrict__ my_ctrl,
                 P2PPeers peers, int my_rank, unsigned* __restrict__ done, double* __restrict__ err_flag) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const u64 epoch = *(volatile u64*)(my_ctrl + 2) + 1;           // stable until the last block bumps it in p2p_root_done
    const u64 flag = epoch & 0xffffffffull;
    bool ok = true;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        store[i] = p2p_gather(store[i], slots, slot_stride, i, peers, my_rank, flag, ok);
    p2p_root_done(ok, epoch, my_ctrl, peers, my_rank, done, err_flag);
}

}  // namespace pipsort
