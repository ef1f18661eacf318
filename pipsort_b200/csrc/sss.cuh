// Stochastic shotgun search with a device-resident search state (sss_postcal.cpp:102-380), on one GPU or on several.
//
// The reference keeps the neighbourhood as vector<vector<int>>, the explored configurations in an
// unordered_map<vector<int>, double> (postcal.h:43-56,98) and scores the unseen neighbours in an OpenMP loop
// (sss_postcal.cpp:223-255).  Here, per iteration, nothing but the current configuration (<= 8 ints) goes to the
// device and nothing but the neighbours' log-likelihoods (n doubles) comes back:
//   sss_lookup_kernel   thread i UNRANKS neighbour i of the current configuration directly (zero ++ minus ++ plus in the
//                       reference's order, sss_postcal.cpp:20-99,166-186), looks it up in an open-addressing hash table
//                       in HBM (key = the sorted union indices packed into 128 bits) and either copies the stored value
//                       or flags the neighbour as unseen; this rank's share of the unseen ones forms a compact batch;
//   score_lane_kernel / score_batch_kernel  (score_lane.cuh / score.cuh) expand + score + accumulate the batch: one
//                       launch per neighbourhood;
//   sss_push_kernel     (several GPUs only) sends the batch's values to the other ranks through the mailboxes of p2p.cuh;
//   sss_insert_kernel   stores every new value in the table (the reference also inserts after its loop, :280-284) and
//                       scatters them to the neighbours' slots;
//   sss_total_kernel    (from the round the convergence rule first reads on) the running total of all ranks.
// The sampling step (three within-group std::discrete_distribution draws and one across groups from
// std::mt19937(12345), sss_postcal.cpp:289-343) stays on the host: it must reproduce libstdc++'s sequence bit for bit,
// and it needs only the n doubles.
#pragma once
#include "common.cuh"
#include "p2p.cuh"

namespace pipsort {

constexpr u64 SSS_OCC = 1ull << 63;      // "slot occupied" bit of the high key word
constexpr int SSS_IDX_BITS = 15;         // per union index (stored as idx + 1): U <= 32766
constexpr int SSS_MAX_U = (1 << SSS_IDX_BITS) - 2;

struct SssTable {
    u64* klo;
    u64* khi;
    double* val;
    u64 mask;                            // capacity - 1 (capacity is a power of two)
};

struct SssCur {                          // the current configuration, sorted ascending (snp_map order)
    int k;
    int g[KMAX];
};

__host__ __device__ inline void sss_key(const int* cfg, int k, u64& lo, u64& hi) {
    lo = 0; hi = SSS_OCC;
    for (int i = 0; i < k; i++) {
        const u64 v = (u64)(cfg[i] + 1);
        if (i < 4) lo |= v << (SSS_IDX_BITS * i);
        else hi |= v << (SSS_IDX_BITS * (i - 4));
    }
}

__host__ __device__ inline u64 sss_hash(u64 lo, u64 hi) {
    u64 x = lo ^ (hi * 0x9e3779b97f4a7c15ull);
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27; x *= 0x94d049bb133111ebull;
    x ^= x >> 31;
    return x;
}

__device__ inline bool sss_find(const SssTable& t, u64 lo, u64 hi, double& v) {
    u64 s = sss_hash(lo, hi) & t.mask;
    for (;;) {
        const u64 h = t.khi[s];
        if (!(h & SSS_OCC)) return false;
        if (h == hi && t.klo[s] == lo) { v = t.val[s]; return true; }
        s = (s + 1) & t.mask;
    }
}

// distinct keys only (every configuration is inserted once); concurrent with other inserts, not with finds
__device__ inline void sss_put(const SssTable& t, u64 lo, u64 hi, double v) {
    u64 s = sss_hash(lo, hi) & t.mask;
    for (;;) {
        const u64 old = atomicCAS(t.khi + s, 0ull, hi);
        if (old == 0ull) { t.klo[s] = lo; t.val[s] = v; return; }
        s = (s + 1) & t.mask;
    }
}

// Sizes of the three neighbourhood groups of a configuration with k of U SNPs (sss_postcal.cpp:20-99)
__host__ __device__ inline void sss_nbd_sizes(int U, int k, int c, long long& nz, long long& nm, long long& np) {
    nz = (long long)(U - k) * k;
    nm = k;
    np = k < c ? (U - k) : 0;
}

// Neighbour i (in zero ++ minus ++ plus order) of cur -> sorted configuration out[0..kk); returns kk.
//   zero : added SNP outer (ascending over the non-members), dropped position inner (ascending)   (:72-99)
//   minus: dropped position ascending                                                            (:50-69)
//   plus : added SNP ascending over the non-members, empty when k >= c                           (:20-48)
__host__ __device__ inline int sss_neighbour(const SssCur& cur, int U, int c, long long i, int* out) {
    long long nz, nm, np;
    sss_nbd_sizes(U, cur.k, c, nz, nm, np);
    int drop = -1, add = -1;
    if (i < nz) { add = (int)(i / cur.k); drop = (int)(i % cur.k); }
    else if (i < nz + nm) drop = (int)(i - nz);
    else add = (int)(i - nz - nm);
    int g = -1;
    if (add >= 0) {                      // the add-th SNP that is not in cur
        g = add;
        for (int j = 0; j < cur.k; j++) if (cur.g[j] <= g) g++;
    }
    int kk = 0;
    bool placed = g < 0;
    for (int j = 0; j < cur.k; j++) {
        if (j == drop) continue;
        if (!placed && g < cur.g[j]) { out[kk++] = g; placed = true; }
        out[kk++] = cur.g[j];
    }
    if (!placed) out[kk++] = g;
    return kk;
}

// ---- the kernels of one round ---------------------------------------------------------------------------------------------
// The neighbourhood may be split over several GPUs (one process per GPU; sss_postcal.cpp:223-255 is the loop being split).
// Every rank runs the whole search in lockstep on a REPLICATED explored-configuration table (same seed, same values, hence
// the same trajectory); of every round's unseen neighbours rank r expands + scores + accumulates those with neighbour index
// i = r (mod world); the max-|l| values travel to every peer through the mailboxes of p2p.cuh (written straight into the
// peer's memory over NVLink); the accumulators stay rank-partial until they are combined (pipsort_p2p_reduce_to_root /
// all-reduce) at the end.  With world = 1 the one rank scores every unseen neighbour and no mailbox is touched.
struct SssShard {
    int world, rank;
    unsigned flag;                               // this round's epoch (low 32 bits), never 0; unused when world = 1
    ulonglong2* peer_slot[P2P_MAX_WORLD];        // [p]: where THIS rank's values go in peer p's mailbox (nullptr for p == rank)
    const ulonglong2* my_slot[P2P_MAX_WORLD];    // [p]: where peer p's values arrive in this rank's mailbox
};

// thread i < n: neighbour i; thread n: the current configuration (scored by rank 0 when unseen, :190-202).  out_l[i] gets the
// stored value of a seen neighbour; unseen ones are flagged (state[i] = 1) on every rank and appended to THIS rank's batch
// when i = rank (mod world) (pos_of[i] = row of the batch).
__global__ void __launch_bounds__(256)
sss_lookup_kernel(SssTable tab, SssCur cur, int U, int c, long long n, int kmax, int world, int rank, double* __restrict__ out_l,
                  int* __restrict__ batch, unsigned char* __restrict__ upd, int* __restrict__ pos_of,
                  unsigned char* __restrict__ state, int* __restrict__ counter /* [0] own batch rows, [1] unseen in total */) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    int cfg[KMAX];
    int kk;
    if (i == n) { kk = cur.k; for (int j = 0; j < kk; j++) cfg[j] = cur.g[j]; }
    else kk = sss_neighbour(cur, U, c, i, cfg);
    u64 lo, hi;
    sss_key(cfg, kk, lo, hi);
    double v = 0.0;
    const bool found = sss_find(tab, lo, hi, v);
    int row = -1;
    if (i == n) {
        // the current configuration is re-scored only when unseen, by rank 0; the other ranks keep row 0 as a no-op
        row = 0;
        upd[0] = (!found && rank == 0) ? 1 : 0;
        if (rank != 0) kk = -1;                                  // all -1: scored as the null configuration WITHOUT updates
    } else {
        state[i] = found ? 0 : 1;
        if (found) { out_l[i] = v; return; }
        atomicAdd(counter + 1, 1);
        if ((int)(i % world) != rank) return;
        const int pos = atomicAdd(counter, 1);
        pos_of[i] = 1 + pos;
        row = 1 + pos;
        upd[row] = 1;
    }
    for (int j = 0; j < kmax; j++) batch[(size_t)row * kmax + j] = j < kk ? cfg[j] : -1;
}

// thread i < n: an unseen neighbour scored by this rank sends its value to every peer (world > 1 only)
__global__ void __launch_bounds__(256)
sss_push_kernel(SssShard sh, long long n, const unsigned char* __restrict__ state, const int* __restrict__ pos_of,
                const double* __restrict__ scored) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !state[i] || (int)(i % sh.world) != sh.rank) return;
    const ulonglong2 w = p2p_encode(scored[pos_of[i]], sh.flag);
    for (int p = 0; p < sh.world; p++)
        if (p != sh.rank) sh.peer_slot[p][i] = w;
}

// thread i < n: every unseen neighbour enters the (replicated) table on every rank, with the value its owner computed (the
// reference also inserts after its loop, :280-284), and goes to the neighbour's slot of out_l
__global__ void __launch_bounds__(256)
sss_insert_kernel(SssTable tab, SssCur cur, int U, int c, long long n, SssShard sh, const unsigned char* __restrict__ state,
                  const int* __restrict__ pos_of, const double* __restrict__ scored, double* __restrict__ out_l,
                  double* __restrict__ err_flag) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !state[i]) return;
    const int owner = (int)(i % sh.world);
    double v;
    if (owner == sh.rank) {
        v = scored[pos_of[i]];
    } else {
        bool ok = true;
        v = p2p_take(sh.my_slot[owner] + i, sh.flag, ok);
        if (!ok) { atomicAdd(err_flag, 1.0); return; }
    }
    int cfg[KMAX];
    const int kk = sss_neighbour(cur, U, c, i, cfg);
    u64 lo, hi;
    sss_key(cfg, kk, lo, hi);
    out_l[i] = v;
    sss_put(tab, lo, hi, v);
}

// The running total (sss_sum_lkl, consulted by the convergence rule from round 100 on, sss_postcal.cpp:265-270), as
// finalize_kernel would report it for the sum of the ranks' stores: every rank sends the bins of its partial total to every
// peer, adds all of them in rank order (so that all ranks see bit-identical sums and take the same branch) and decodes the
// sums like any accumulator.  One warp.
__global__ void __launch_bounds__(32)
sss_total_kernel(AccDev acc, SssShard sh, long long off, double cx, double* __restrict__ out_total, double* __restrict__ err_flag) {
    const int lane = threadIdx.x;
    const double* own = bin_ptr(acc, SCAL, S_TOTAL);
    for (int t = lane; t < acc.NB; t += 32) {
        const ulonglong2 w = p2p_encode(own[(size_t)t * acc.Upad], sh.flag);
        for (int p = 0; p < sh.world; p++)
            if (p != sh.rank) sh.peer_slot[p][off + t] = w;
    }
    bool ok = true;
    auto bin = [&](int t) {                      // bin t of the total, summed over the ranks
        double v = 0.0;
        for (int p = 0; p < sh.world; p++)
            v += p == sh.rank ? own[(size_t)t * acc.Upad] : p2p_take(sh.my_slot[p] + off + t, sh.flag, ok);
        return v;
    };
    int top = -1;
    for (int t = lane; t < acc.NB; t += 32)
        if (bin(t) > 0.0) top = t;
    top = __reduce_max_sync(0xffffffffu, top);
    if (__any_sync(0xffffffffu, !ok)) {          // a peer's bins did not arrive: the search reports the error when it ends
        if (lane == 0) atomicAdd(err_flag, 1.0);
        return;
    }
    if (lane == 0) {                             // (the peers' words of these bins have arrived: bin() reads them at once)
        const XAcc x = top < 0 ? xacc_empty() : bins_decode(top, acc.bias, [&](int k) { return bin(top - k); });
        *out_total = xlog_or_zero(x, cx);
    }
}

__global__ void __launch_bounds__(256) sss_rehash_kernel(SssTable from, SssTable to) {
    const u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (s > from.mask) return;
    const u64 h = from.khi[s];
    if (h & SSS_OCC) sss_put(to, from.klo[s], h, from.val[s]);
}

}  // namespace pipsort
