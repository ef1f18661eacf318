// pipsort_b200 engine: host side of the C-ABI declared in include/pipsort_b200.h.
//
// Owns the device copy of one locus, the accumulator store and a CUDA stream; launches the kernels in
// score.cuh (generic, warp per union configuration) and exhaustive.cuh (register kernel, lane per
// union subset).  No CPU compute path exists: without a usable CUDA device every entry point fails.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <numeric>
#include <random>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pipsort_b200.h"
#include "common.cuh"
#include "exhaustive.cuh"
#include "given.cuh"
#include "prep.cuh"
#include "sss.cuh"
#include "p2p.cuh"
#include "score.cuh"
#include "score_lane.cuh"

using namespace pipsort;

#define PIPSORT_INTERNAL_NO_UPLOAD_WAIT 0x80000000u   /* not part of the public flag set */
#define PIPSORT_INTERNAL_WITH_PAIRS 0x40000000u       /* build the WP tables of the exhaustive kernel in pipsort_create's own launch */

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t err__ = (call);                                                                \
        if (err__ != cudaSuccess)                                                                  \
            return fail(PIPSORT_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), __FILE__, __LINE__); \
    } while (0)

u64 binom_host(int n, int k, bool* overflow) {
    if (k < 0 || k > n) return 0;
    unsigned __int128 v = 1;
    for (int i = 1; i <= k; i++) {
        v = v * (unsigned)(n - k + i) / (unsigned)i;
        if (v >> 63) { if (overflow) *overflow = true; return ~0ull >> 1; }
    }
    return (u64)v;
}

// ---- preparation kernels ------------------------------------------------------------------------------
// W[i][j] = d * sigma[orig[i]][orig[j]]  (permutation into the internal order + the d_s scaling of construct_diagC's
// diagonal, postcal.cpp:89,250,254-255) and the per-SNP vectors A = 1 + W_ii, z, 1/A, z/A, E_s({i}) = e1m 2^e1n,
// for BOTH studies in one launch (blockIdx.z = study): a locus that takes 60 us to evaluate should not
// spend 20 us on four tiny preparation launches.  Thread j == 0 of row i also fills the per-SNP vectors of i.
struct PrepStudyArgs {
    const double* sigma; const double* z_raw; const int* orig;
    int n_raw, n, ldw;
    double d;
    double *W, *A, *z, *invA, *u, *e1m;
    int* e1n;
    double2* WP;     // (n + 1) x ldp table { W_ij, E{i,j} } of the exhaustive kernel, or nullptr: built later, on demand
    int ldp;
};
struct PrepLocusArgs { PrepStudyArgs s[2]; };

__global__ void __launch_bounds__(128) prepare_locus_kernel(PrepLocusArgs P) {
    const PrepStudyArgs& S = P.s[blockIdx.z];
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y;
    if (i > S.n || (i == S.n && !S.WP)) return;
    if (i == S.n) {                                            // the all-zero row of the WP table
        if (j < S.ldp) S.WP[(size_t)i * S.ldp + j] = make_double2(0.0, 0.0);
        return;
    }
    const int oi = S.orig[i];
    double v = 0.0;
    if (j < S.n) v = S.d * S.sigma[(size_t)oi * S.n_raw + S.orig[j]];
    if (j < S.ldw) S.W[(size_t)i * S.ldw + j] = v;
    if (j != 0 && !S.WP) return;
    // the per-SNP values of i: stored by thread j == 0; every thread of the row needs them for its table entry (computing them
    // per thread -- one exp -- costs less than a second launch that reads them back: a 150-SNP locus is 38 us of evaluation)
    const double a = 1.0 + S.d * S.sigma[(size_t)oi * S.n_raw + oi];
    const double zi = S.z_raw[oi];
    const double invA = 1.0 / a, u = zi / a;
    double m;
    int e;
    xexp(0.5 * S.d * (zi * zi / a), m, e);
    const double e1m = m / sqrt(a);
    if (j == 0) {
        S.A[i] = a;
        S.z[i] = zi;
        S.invA[i] = invA;
        S.u[i] = u;
        S.e1m[i] = e1m;
        S.e1n[i] = e;
    }
    if (S.WP && j < S.ldp) {
        double2 w = make_double2(0.0, 0.0);                    // columns >= n: the absent SNP
        if (j < S.n) {
            w.x = v;
            if (j != i) {
                const int oj = S.orig[j];
                w.y = pair_entry(0.5 * S.d, e1m, e, invA, u, v, 1.0 + S.d * S.sigma[(size_t)oj * S.n_raw + oj], S.z_raw[oj]);
            }
        }
        S.WP[(size_t)i * S.ldp + j] = w;
    }
}

struct PairTablesArgs { StudyDev st[2]; double2* WP[2]; };
__global__ void __launch_bounds__(128) pair_tables_kernel(PairTablesArgs T) {   // WP table (common.cuh) of both studies
    const StudyDev& S = T.st[blockIdx.z];
    double2* __restrict__ WP = T.WP[blockIdx.z];
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y;
    if (j >= S.ldp || i > S.n) return;
    double2 v = make_double2(0.0, 0.0);                  // row n, columns >= n: the absent SNP
    if (i < S.n && j < S.n) v = make_double2(S.W[(size_t)i * S.ldw + j], pair_table_entry(S, i, j));
    WP[(size_t)i * S.ldp + j] = v;
}

// ---- finalize: bins -> log-space results --------------------------------------------------------------
// warp-collective: lanes scan the bins of one accumulator in parallel, the top three non-empty bins give M 2^N;
// clear: leave the accumulator empty behind (the finalize kernel then doubles as the reset of the next pass)
__device__ inline XAcc bins_read_warp(const AccDev& a, int slot, int g, int lane, bool clear = false) {
    double* p = bin_ptr(a, slot, g);
    int top = -1;
    for (int b = lane; b < a.NB; b += 32)
        if (p[(size_t)b * a.Upad] > 0.0) top = b;
    top = __reduce_max_sync(0xffffffffu, top);
    if (top < 0) return xacc_empty();
    const XAcc x = bins_decode(top, a.bias, [&](int k) { return p[(size_t)(top - k) * a.Upad]; });
    if (clear) {
        __syncwarp();
        for (int b = lane; b < a.NB; b += 32) p[(size_t)b * a.Upad] = 0.0;
    }
    return x;
}

// The same from registers when the accumulator has at most 32 bins: lane b holds bin b (all the loads of a SNP's five
// accumulators are then issued together -- one memory round trip instead of ten dependent ones).
__device__ inline XAcc bins_from_lanes(double v, int bias) {
    const unsigned mask = __ballot_sync(0xffffffffu, v > 0.0);
    if (!mask) return xacc_empty();
    const int top = 31 - __clz(mask);
    const double m0 = __shfl_sync(0xffffffffu, v, top);
    const double m1 = __shfl_sync(0xffffffffu, v, max(top - 1, 0)), m2 = __shfl_sync(0xffffffffu, v, max(top - 2, 0));
    return bins_decode(top, bias, [&](int k) { return k == 0 ? m0 : (k == 1 ? m1 : m2); });
}

// res: [0] total, [1] noCausal[0], [2] noCausal[1], then 5 arrays of U (internal order):
//      postValues study 0, postValues study 1, sharedPips, sharedLL, notSharedLL
// One warp per union SNP (plus one warp per scalar).
constexpr int FIN_WARPS = 8;
__global__ void __launch_bounds__(FIN_WARPS * 32) finalize_kernel(AccDev acc, int U, double cx, double cy, double* __restrict__ res,
                                                                  int clear) {
    // launched with programmatic stream serialization: the blocks may become resident while the kernel before them in
    // the stream is still draining; nothing of the accumulator store is touched before that kernel has completed
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * FIN_WARPS + (threadIdx.x >> 5);
    if (blockIdx.x == 0 && threadIdx.x < NCOUNTER) {
        res[3 + (size_t)5 * U + threadIdx.x] = acc.counters[threadIdx.x];
        if (clear) acc.counters[threadIdx.x] = 0.0;
    }
    if (w < 3) {
        const XAcc v = bins_read_warp(acc, SCAL, w, lane, clear != 0);
        if (lane == 0) res[w] = xlog_or_zero(v, cx);
        return;
    }
    const int g = w - 3;
    if (g >= U) return;
    XAcc x1, x2, x3, ys, yn;
    if (acc.NB <= 32) {
        double v[5];
#pragma unroll
        for (int k = 0; k < 5; k++) {   // X1 X2 X3 YS YN
            double* q = bin_ptr(acc, k, g) + (size_t)lane * acc.Upad;
            v[k] = lane < acc.NB ? *q : 0.0;
            if (clear && lane < acc.NB && v[k] != 0.0) *q = 0.0;
        }
        x1 = bins_from_lanes(v[X1], acc.bias); x2 = bins_from_lanes(v[X2], acc.bias); x3 = bins_from_lanes(v[X3], acc.bias);
        ys = bins_from_lanes(v[YS], acc.bias); yn = bins_from_lanes(v[YN], acc.bias);
    } else {
        x1 = bins_read_warp(acc, X1, g, lane, clear != 0); x2 = bins_read_warp(acc, X2, g, lane, clear != 0);
        x3 = bins_read_warp(acc, X3, g, lane, clear != 0);
        ys = bins_read_warp(acc, YS, g, lane, clear != 0); yn = bins_read_warp(acc, YN, g, lane, clear != 0);
    }
    if (lane >= 5) return;
    XAcc p0 = x1, p1 = x2;
    xmerge(p0, x3);
    xmerge(p1, x3);
    // five logarithms: one lane each
    const XAcc mine = lane == 0 ? p0 : (lane == 1 ? p1 : (lane == 2 ? x3 : (lane == 3 ? ys : yn)));
    res[3 + (size_t)lane * U + g] = xlog_or_zero(mine, lane < 3 ? cx : cy);
}

// Layout of one prior of the grid read: pi'(J,a) as a (KMAX+1) x (KMAX+1) table (row J), then cx = -K/2 + U log(1-gamma).
constexpr int PRIOR_STRIDE = (KMAX + 1) * (KMAX + 1) + 1;

// class slot / scalar of the class-resolved store (common.cuh) read by ONE lane: the top three non-empty bins, as bins_read_warp
__device__ inline XAcc bins_read_lane(const AccDev& a, int slot, int g, bool clear) {
    double* p = bin_ptr(a, slot, g);
    int top = -1;
    for (int b = 0; b < a.NB; b++)
        if (p[(size_t)b * a.Upad] > 0.0) top = b;
    if (top < 0) return xacc_empty();
    const XAcc x = bins_decode(top, a.bias, [&](int k) { return p[(size_t)(top - k) * a.Upad]; });
    if (clear)
        for (int b = 0; b <= top; b++) p[(size_t)b * a.Upad] = 0.0;
    return x;
}

// acc += w * v  (w >= 0 a prior weight; a zero weight or an empty v adds nothing)
__device__ __forceinline__ void xadd_weighted(XAcc& acc, const XAcc& v, double w) {
    const double m = v.M * w;
    if (m > 0.0) xadd(acc, m, v.N);
}

// Finalize of the class-resolved store (PIPSORT_PRIOR_CLASSES, DESIGN.md section 5f) for n_priors priors: prior i is
// pri[i * PRIOR_STRIDE ..] (PRIOR_STRIDE above) and its results go to res[i * (3 + 5 U) ..] in finalize_kernel's layout; the
// counters follow the last prior (the same for every prior).  One warp per scalar output / union SNP: lane l reads the class
// slots l, l + 32, .. once, then every prior costs one weighted warp sum per output.
constexpr int GRID_LANE_SLOTS = (cls_nslot(KMAX) + 31) / 32;
__global__ void __launch_bounds__(FIN_WARPS * 32) finalize_grid_kernel(AccDev acc, int U, int n_priors, const double* __restrict__ pri,
                                                                       double cy, double* __restrict__ res, int clear) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * FIN_WARPS + (threadIdx.x >> 5);
    const int C = acc.ccls;
    const size_t stride = 3 + (size_t)5 * U;
    if (blockIdx.x == 0 && threadIdx.x < NCOUNTER) {
        res[(size_t)n_priors * stride + threadIdx.x] = acc.counters[threadIdx.x];
        if (clear) acc.counters[threadIdx.x] = 0.0;
    }
    if (w < 3) {   // total: T[J][a], weight pi'(J,a);  noCausal[s]: N_s[J], weight pi'(J,0)
        const int n = w == 0 ? (C + 1) * (C + 2) / 2 : C + 1;
        XAcc v[2];
        int row[2];
        for (int q = 0; q < 2; q++) {
            const int k = lane + 32 * q;
            v[q] = xacc_empty();
            row[q] = -1;
            if (k >= n) continue;
            int J = 0, a = k;
            if (w == 0) while (a > J) { J++; a -= J; }
            else { J = k; a = 0; }
            const int idx = w == 0 ? cls_T(J, a) : cls_N(C, w - 1, J);
            v[q] = bins_read_lane(acc, cls_nslot(C) + idx / acc.Upad, idx % acc.Upad, clear != 0);
            row[q] = J * (KMAX + 1) + a;
        }
        for (int i = 0; i < n_priors; i++) {
            const double* pi = pri + (size_t)i * PRIOR_STRIDE;
            XAcc s = xacc_empty();
            for (int q = 0; q < 2; q++)
                if (row[q] >= 0) xadd_weighted(s, v[q], pi[row[q]]);
            s = xwarp_sum(s);
            if (lane == 0) res[(size_t)i * stride + w] = xlog_or_zero(s, pi[PRIOR_STRIDE - 1]);
        }
        return;
    }
    const int g = w - 3;
    if (g >= U) return;
    XAcc v[GRID_LANE_SLOTS];
    int row[GRID_LANE_SLOTS], st[GRID_LANE_SLOTS];
    XAcc ys = xacc_empty(), yn = xacc_empty();      // likelihood-only sums: the same for every prior
#pragma unroll
    for (int q = 0; q < GRID_LANE_SLOTS; q++) {
        const int k = lane + 32 * q;
        v[q] = xacc_empty();
        row[q] = 0; st[q] = -1;
        if (k >= cls_nslot(C)) continue;
        int J = 1, r = k;
        while (r >= 3 * J) { r -= 3 * J; J++; }
        const int t = r / J, ap = r - t * J;
        v[q] = bins_read_lane(acc, k, g, clear != 0);
        st[q] = t;
        row[q] = J * (KMAX + 1) + ap + (t == 2 ? 1 : 0);
        if (v[q].M > 0.0) xadd(t == 2 ? ys : yn, v[q].M, v[q].N);
    }
    ys = xwarp_sum(ys);
    yn = xwarp_sum(yn);
    if (lane == 0) {
        res[3 + (size_t)3 * U + g] = xlog_or_zero(ys, cy);
        res[3 + (size_t)4 * U + g] = xlog_or_zero(yn, cy);
    }
    for (int i = 0; i < n_priors; i++) {
        const double* pi = pri + (size_t)i * PRIOR_STRIDE;
        XAcc x[3] = {xacc_empty(), xacc_empty(), xacc_empty()};
#pragma unroll
        for (int q = 0; q < GRID_LANE_SLOTS; q++) {
            if (st[q] < 0) continue;
            const double wq = pi[row[q]];
            if (st[q] == 0) xadd_weighted(x[0], v[q], wq);
            else if (st[q] == 1) xadd_weighted(x[1], v[q], wq);
            else xadd_weighted(x[2], v[q], wq);
        }
#pragma unroll
        for (int t = 0; t < 3; t++) x[t] = xwarp_sum(x[t]);
        XAcc p0 = x[0], p1 = x[1];
        xmerge(p0, x[2]);
        xmerge(p1, x[2]);
        const double cx = pi[PRIOR_STRIDE - 1];
        double* r = res + (size_t)i * stride + 3;
        if (lane == 0) r[g] = xlog_or_zero(p0, cx);
        else if (lane == 1) r[(size_t)U + g] = xlog_or_zero(p1, cx);
        else if (lane == 2) r[(size_t)2 * U + g] = xlog_or_zero(x[2], cx);
        else if (lane == 3 && i > 0) { r[(size_t)3 * U + g] = xlog_or_zero(ys, cy); r[(size_t)4 * U + g] = xlog_or_zero(yn, cy); }
    }
}

// The root's half of the multi-GPU combine step fused with the finalize (accumulators of at most 32 bins): lane b of the warp
// of a SNP takes bin b of the SNP's five accumulators from the root's own store AND from every peer's mailbox slot (polling
// each element until it carries this epoch's flag, p2p.cuh), so the sum over the GPUs never goes back to memory; the root's
// store is left empty.  The last block posts `consumed` to the peers.  Replaces p2p_merge_kernel + finalize_kernel.
__global__ void __launch_bounds__(FIN_WARPS * 32)
finalize_merge_kernel(AccDev acc, int U, double cx, double cy, double* __restrict__ res, const ulonglong2* slots, size_t slot_stride,
                      size_t bins_len, u64* __restrict__ my_ctrl, P2PPeers peers, int my_rank, unsigned* __restrict__ done,
                      double* __restrict__ err_flag) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const u64 epoch = *(volatile u64*)(my_ctrl + 2) + 1;           // stable until the last block bumps it below
    const u64 flag = epoch & 0xffffffffull;
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * FIN_WARPS + (threadIdx.x >> 5);
    bool ok = true;
    auto take = [&](size_t idx) -> double {                        // element idx of the store, summed over all GPUs; own copy cleared
        double v = acc.bins[idx];
        if (v != 0.0) acc.bins[idx] = 0.0;
        if (peers.world <= 8) {
            // all peers' copies are requested at once (one round trip, not one per peer: with 7 peers the serial polls were
            // most of the step at N = 8), re-requested until each carries this epoch's flag, then added in rank order
            ulonglong2 wr[8];
            unsigned pend = 0;
#pragma unroll
            for (int r = 0; r < 8; r++)
                if (r < peers.world && r != my_rank) {
                    wr[r] = p2p_load(slots + (size_t)r * slot_stride + idx);
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
                    if (pend >> r & 1) wr[r] = p2p_load(slots + (size_t)r * slot_stride + idx);
            }
#pragma unroll
            for (int r = 0; r < 8; r++)
                if (r < peers.world && r != my_rank) v += p2p_decode(wr[r]);
            return v;
        }
        for (int r = 0; r < peers.world; r++)
            if (r != my_rank) v += p2p_take(slots + (size_t)r * slot_stride + idx, flag, ok);
        return v;
    };
    if (blockIdx.x == 0 && threadIdx.x < NCOUNTER) res[3 + (size_t)5 * U + threadIdx.x] = take(bins_len - NCOUNTER + threadIdx.x);
    if (w < 3) {
        const double v = lane < acc.NB ? take(((size_t)SCAL * acc.NB + lane) * acc.Upad + w) : 0.0;
        const XAcc x = bins_from_lanes(v, acc.bias);
        if (lane == 0) res[w] = xlog_or_zero(x, cx);
    } else if (w - 3 < U) {
        const int g = w - 3;
        double v[5];
#pragma unroll
        for (int k = 0; k < 5; k++) v[k] = lane < acc.NB ? take(((size_t)k * acc.NB + lane) * acc.Upad + g) : 0.0;
        const XAcc x1 = bins_from_lanes(v[X1], acc.bias), x2 = bins_from_lanes(v[X2], acc.bias), x3 = bins_from_lanes(v[X3], acc.bias);
        const XAcc ys = bins_from_lanes(v[YS], acc.bias), yn = bins_from_lanes(v[YN], acc.bias);
        if (lane < 5) {
            XAcc p0 = x1, p1 = x2;
            xmerge(p0, x3);
            xmerge(p1, x3);
            const XAcc mine = lane == 0 ? p0 : (lane == 1 ? p1 : (lane == 2 ? x3 : (lane == 3 ? ys : yn)));
            res[3 + (size_t)lane * U + g] = xlog_or_zero(mine, lane < 3 ? cx : cy);
        }
    }
    if (!ok) atomicAdd(err_flag, 1.0);
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned d = atomicAdd(done, 1u);
        if (d == gridDim.x - 1) {                    // every block has read the slots: the peers may overwrite them
            *done = 0;
            my_ctrl[2] = epoch;
            __threadfence_system();
            for (int r = 0; r < peers.world; r++)
                if (r != my_rank) *(volatile u64*)(peers.ctrl[r] + 1) = epoch;
        }
    }
}

__global__ void add_bins_kernel(double* __restrict__ dst, const double* __restrict__ src, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += src[i];
}

// ---- FP64 peak micro-benchmark ------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double a, double b) {
    double x0 = threadIdx.x * 1e-9, x1 = x0 + 1e-9, x2 = x0 + 2e-9, x3 = x0 + 3e-9, x4 = x0 + 4e-9, x5 = x0 + 5e-9,
           x6 = x0 + 6e-9, x7 = x0 + 7e-9;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 12345.678) out[0] = s;   // never true in practice; keeps the chains alive
}

}  // namespace

struct pipsort_engine {
    int device = 0;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    char* l2_scratch = nullptr;
    size_t cap_l2 = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr, ev_up = nullptr;
    bool evk_valid = false;
    LocusDev L, L_host_copy;
    LocusDev* d_L = nullptr;        // device copy (the slow path of the register kernel reads it by pointer)
    int U = 0, kb = 3, sm_count = 148;
    int n_raw[2] = {0, 0};
    double K = 0, gamma = 0, p = 0;
    std::vector<int> perm;          // internal -> user union index
    std::vector<int> orig[2];       // study-local (internal order) -> original study index
    std::vector<int> loc[2];        // internal union index -> study-local index or -1
    std::vector<int> types;         // internal union index -> 0 shared, 1 only study 0, 2 only study 1, 3 nowhere
    struct Alloc { void* p; bool pinned; };
    std::vector<Alloc> allocs;      // what did not come from the arena: device pool buffers and pinned host buffers
    char* pin = nullptr;            // pinned staging buffer of the stream kit (PIN_BYTES), bump-allocated, never reused
    size_t pin_off = 0;             // within an engine's life: an asynchronous copy may still be reading a slice
    bool defer_upload_sync = false; // one-call path: the caller's buffers outlive the call, no wait after the uploads
    char* arena = nullptr;          // one allocation for (nearly) all device arrays of the engine
    size_t arena_cap = 0, arena_off = 0;
    int* d_snp_map = nullptr;       // user order, [2][U]
    double* d_res = nullptr;
    std::vector<double> h_res;
    double* h_res_pin = nullptr;    // slice of the pinned staging buffer for the result read-back
    size_t bins_len = 0;
    u64 launches = 0;
    // scratch of pipsort_score_union_configs (callers with host buffers)
    int* d_idx = nullptr; unsigned char* d_upd = nullptr; double* d_out = nullptr;
    size_t cap_idx = 0, cap_upd = 0, cap_out = 0;
    int score_smem_set = 0;
    bool lane_smem_set = false;
    ExhScratch exh;
    bool use_reg_kernel = true;
    ExhCostModel cost_model;           // step costs of the exhaustive kernel from the SNP-type layout (plan + shard boundaries)
    bool capturing = false;
    std::vector<cudaGraphExec_t> graphs;
    uint64_t last_read_count = 0;   // configuration count seen by the last pipsort_read_accumulators
    // stochastic shotgun search state (pipsort_sss): explored-configuration hash table + per-iteration buffers
    struct Sss {
        SssTable tab{nullptr, nullptr, nullptr, 0};
        u64 count = 0;              // entries in the table
        double* d_out_l = nullptr; int* d_batch = nullptr; unsigned char* d_upd = nullptr; int* d_counter = nullptr;
        double* d_scored = nullptr; unsigned char* d_state = nullptr; int* d_pos_of = nullptr; double* d_total = nullptr;
        double* h_out_l = nullptr;  // pinned: [n_max] neighbour values, [n_max + 1] the running total
        size_t cap_out_l = 0, cap_batch = 0, cap_upd = 0, cap_counter = 0, cap_scored = 0, cap_state = 0, cap_pos_of = 0,
               cap_total = 0, cap_h_out_l = 0;
    } sss;
    // peer-memory combine (p2p.cuh): this rank's mailbox + the peers' mapped mailboxes
    struct P2P {
        double* mailbox = nullptr;   // 256-byte header (8 control words) | world slots (16 bytes per accumulator double)
        unsigned* d_done = nullptr;
        void* peer_base[P2P_MAX_WORLD] = {nullptr};
        P2PPeers peers;
        int world = 0, rank = 0, root = 0;
        int cache_slot = -1;         // entry of the process-wide mailbox cache this engine has borrowed
        u64* sss_epoch = nullptr;    // rounds of the sharded search on this mailbox (lives with the mailbox, not the engine)
        bool connected = false;
    } p2p;
    PrepResult prep[2];             // PIPSORT_RAW_LD: what the on-device pre-processing found per study
    bool prepped = false;
    // PIPSORT_PRIOR_CLASSES: the store is class-resolved (AccDev::ccls > 0); the engine's own prior as the grid finalize reads it
    bool classes = false;
    double* d_own_prior = nullptr;  // [PRIOR_STRIDE]
    double* d_grid = nullptr;       // grid read: priors | results | counters
    size_t cap_grid = 0;
    std::vector<double> h_grid;
};

namespace {

// Stream-ordered allocation from the device's default memory pool: after the first engine on a device the
// pool serves create/destroy without touching the driver allocator (the locus arrays of a fine-mapping run
// are created and destroyed once per locus).
// Streams and timing events are recycled across engines of one process (a fine-mapping run creates and destroys one
// engine per locus; cudaStreamCreate / cudaEventCreate are a measurable part of a 0.1 ms locus).
constexpr size_t PIN_BYTES = (size_t)256 << 10;   // pinned staging per kit: small uploads / the result read-back go through it
struct StreamKit { cudaStream_t stream; cudaEvent_t ev[5]; char* pin; };
std::vector<StreamKit>& kit_cache(int device) {
    static std::vector<StreamKit> cache[64];
    return cache[device & 63];
}
std::mutex& kit_mutex() { static std::mutex m; return m; }

int kit_acquire(int device, StreamKit* k) {
    {
        std::lock_guard<std::mutex> g(kit_mutex());
        auto& c = kit_cache(device);
        if (!c.empty()) { *k = c.back(); c.pop_back(); return 0; }
    }
    *k = StreamKit{};
    cudaError_t err = cudaStreamCreateWithFlags(&k->stream, cudaStreamNonBlocking);
    for (int i = 0; i < 5 && err == cudaSuccess; i++) err = cudaEventCreateWithFlags(&k->ev[i], i < 4 ? cudaEventDefault : cudaEventDisableTiming);
    if (err != cudaSuccess) {   // a kit is complete or not at all
        for (cudaEvent_t ev : k->ev) if (ev) cudaEventDestroy(ev);
        if (k->stream) cudaStreamDestroy(k->stream);
        return fail(PIPSORT_E_CUDA, "stream / event creation failed: %s", cudaGetErrorString(err));
    }
    if (cudaHostAlloc((void**)&k->pin, PIN_BYTES, cudaHostAllocDefault) != cudaSuccess) { k->pin = nullptr; cudaGetLastError(); }
    return 0;
}
void kit_release(int device, const StreamKit& k) {
    std::lock_guard<std::mutex> g(kit_mutex());
    kit_cache(device).push_back(k);
}

// one-time, per-process initialisations (device count, SM counts, pool thresholds, expansion tables, occupancy) may be
// reached by several host threads creating their first engines at once: they all run under this mutex
std::mutex& init_mutex() { static std::mutex m; return m; }

int pool_setup(int device) {
    static bool done[64] = {false};
    std::lock_guard<std::mutex> g(init_mutex());
    if (device < 64 && done[device]) return 0;
    cudaMemPool_t pool;
    CU(cudaDeviceGetDefaultMemPool(&pool, device));
    unsigned long long keep = ~0ull;
    CU(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    if (device < 64) done[device] = true;
    return 0;
}

// Device memory of an engine comes from ONE stream-ordered allocation made in pipsort_create (an arena with a bump
// pointer): a locus needs ~25 arrays, and 25 cudaMallocAsync / cudaFreeAsync pairs are a visible part of a 0.3 ms
// create-run-read-destroy cycle.  Requests the arena cannot hold (its size is an estimate) fall back to the pool.  Every
// buffer of an engine comes from dev_alloc or grow and goes back in release or pipsort_destroy; nothing is allocated while
// a graph is being captured (its replays could not run until such a buffer were freed, and destroy would free it outside
// the graph).
const char* const CAPTURE_NO_ALLOC = "run the pass once before capturing it (the first run allocates what the pass needs)";

// where a buffer may come from: the arena (then the pool when it is full), the pool only, pinned host memory
enum class Mem { arena, pool, pinned };

template <class T>
int dev_alloc(pipsort_engine* e, T** p, size_t count, Mem where = Mem::arena) {
    const size_t bytes = (std::max<size_t>(count, 1) * sizeof(T) + 255) & ~(size_t)255;
    if (where == Mem::arena && e->arena && e->arena_off + bytes <= e->arena_cap) {
        *p = reinterpret_cast<T*>(e->arena + e->arena_off);
        e->arena_off += bytes;
        return 0;
    }
    if (e->capturing) return fail(PIPSORT_E_ARG, "%s", CAPTURE_NO_ALLOC);
    void* q = nullptr;
    const bool pinned = where == Mem::pinned;
    const cudaError_t err = pinned ? cudaMallocHost(&q, bytes) : cudaMallocAsync(&q, bytes, e->stream);
    if (err != cudaSuccess) {
        cudaGetLastError();                  // a refused request leaves no error pending for the engine's next call
        return fail(PIPSORT_E_CUDA, "allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(err));
    }
    e->allocs.push_back({q, pinned});
    *p = static_cast<T*>(q);
    return 0;
}

// frees a buffer from dev_alloc (stream-ordered; an arena slice stays where it is) and nulls the pointer
template <class T>
int release(pipsort_engine* e, T** p) {
    void* q = *p;
    *p = nullptr;
    for (size_t i = 0; i < e->allocs.size(); i++) {
        if (e->allocs[i].p != q) continue;
        const bool pinned = e->allocs[i].pinned;
        e->allocs.erase(e->allocs.begin() + i);
        CU(pinned ? cudaFreeHost(q) : cudaFreeAsync(q, e->stream));
        break;
    }
    return 0;
}

// a buffer of at least n elements in *p: keeps it when *cap >= n, else replaces it; on failure *p is null and *cap 0.
// Buffers that grow on demand come from the pool (or pinned memory), never from the arena: the arena's room is for the locus.
template <class T>
int grow(pipsort_engine* e, T** p, size_t* cap, size_t n, Mem where = Mem::pool) {
    if (*cap >= n) return 0;
    if (e->capturing) return fail(PIPSORT_E_ARG, "%s", CAPTURE_NO_ALLOC);
    *cap = 0;
    int rc = release(e, p);
    if (!rc) rc = dev_alloc(e, p, n, where);   // sets *p only when it succeeds
    if (!rc) *cap = n;
    return rc;
}

template <class T>
int dev_upload(pipsort_engine* e, T** p, const T* src, size_t count) {
    int rc = dev_alloc(e, p, count);
    if (rc) return rc;
    if (count) CU(cudaMemcpyAsync(*p, src, count * sizeof(T), cudaMemcpyHostToDevice, e->stream));
    return 0;
}

// a slice of the pinned staging buffer, or nullptr when it is used up (callers then copy from pageable memory)
char* pin_slice(pipsort_engine* e, size_t bytes) {
    bytes = (bytes + 63) & ~(size_t)63;
    if (!e->pin || e->pin_off + bytes > PIN_BYTES) return nullptr;
    char* p = e->pin + e->pin_off;
    e->pin_off += bytes;
    return p;
}

// host -> device copy of a small host array that may disappear after the call: staged through pinned memory so that the
// copy is truly asynchronous (a pageable source makes cudaMemcpyAsync block for several microseconds each time)
int upload_small(pipsort_engine* e, void* dst, const void* src, size_t bytes) {
    if (!bytes) return 0;
    if (char* st = pin_slice(e, bytes)) { memcpy(st, src, bytes); src = st; }
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, e->stream));
    return 0;
}

int ensure_score_smem(pipsort_engine* e, int ws_kmax, size_t* bytes) {
    *bytes = SCORE_WARPS * warp_ws_bytes(ws_kmax);
    if (e->score_smem_set < ws_kmax) {
        size_t mx = SCORE_WARPS * warp_ws_bytes(KMAX);
        CU(cudaFuncSetAttribute(score_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mx));
        CU(cudaFuncSetAttribute(exhaustive_generic_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mx));
        CU(cudaFuncSetAttribute(exhaustive_generic_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mx));
        e->score_smem_set = KMAX;
    }
    return 0;
}

// number of expanded configurations of the subsets of size j whose smallest element is g, and of all
// subsets of size j -- by elementary symmetric polynomials of the per-SNP state counts (3 / 1 / 0).
struct WorkModel {
    std::vector<std::vector<double>> E;  // E[m][g] = e_m(w_g .. w_{U-1})
    std::vector<double> w;
    int U;
    WorkModel(const std::vector<int>& types, int c) : U((int)types.size()) {
        w.resize(U);
        for (int g = 0; g < U; g++) w[g] = types[g] == 0 ? 3.0 : (types[g] == 3 ? 0.0 : 1.0);
        E.assign(c + 1, std::vector<double>(U + 1, 0.0));
        for (int g = 0; g <= U; g++) E[0][g] = 1.0;
        for (int m = 1; m <= c; m++)
            for (int g = U - 1; g >= 0; g--) E[m][g] = E[m][g + 1] + w[g] * E[m - 1][g + 1];
    }
    double configs_first(int j, int g) const { return j == 0 ? 1.0 : w[g] * E[j - 1][g + 1]; }
};

// ---- mailboxes of the peer-memory combine step (p2p.cuh), cached per process ----------------------------------------------
// A fine-mapping run creates one engine per locus; cudaMalloc + IPC export + the peers' cudaIpcOpenMemHandle cost far more
// than evaluating a 150-SNP locus.  Mailboxes therefore belong to the process: an engine borrows one that is large enough
// (or allocates it) and hands it back at destroy; peers' mappings are opened once per distinct handle and kept.  The
// control words sit in a fixed header at the START of the mailbox, so epochs and flow control carry over from one engine
// to the next whatever their slot size (slot contents are self-validating by epoch: stale data never matches).
constexpr size_t P2P_HDR_BYTES = 256;
struct MailboxEntry {
    int device, world;
    double* mailbox; size_t bytes; unsigned* d_done;
    u64 sss_epoch;
    bool in_use;
};
std::vector<MailboxEntry*>& mailbox_cache() { static std::vector<MailboxEntry*> c; return c; }
std::mutex& mailbox_mutex() { static std::mutex m; return m; }

int mailbox_acquire(int device, int world, size_t bytes, int* slot) {
    std::lock_guard<std::mutex> g(mailbox_mutex());
    auto& c = mailbox_cache();
    for (size_t i = 0; i < c.size(); i++)
        if (!c[i]->in_use && c[i]->device == device && c[i]->world == world && c[i]->bytes >= bytes) { c[i]->in_use = true; *slot = (int)i; return 0; }
    MailboxEntry m{device, world, nullptr, bytes + bytes / 2, nullptr, 0, true};
    cudaError_t err = cudaMalloc(&m.mailbox, m.bytes);       // cudaMalloc (not the pool): CUDA IPC needs it
    if (err == cudaSuccess) err = cudaMemset(m.mailbox, 0, m.bytes);
    if (err == cudaSuccess) err = cudaMalloc(&m.d_done, sizeof(unsigned));
    if (err == cudaSuccess) err = cudaMemset(m.d_done, 0, sizeof(unsigned));
    if (err != cudaSuccess) {
        if (m.mailbox) cudaFree(m.mailbox);
        if (m.d_done) cudaFree(m.d_done);
        return fail(PIPSORT_E_CUDA, "mailbox allocation failed: %s", cudaGetErrorString(err));
    }
    c.push_back(new MailboxEntry(m));
    *slot = (int)c.size() - 1;
    return 0;
}
void mailbox_release(int slot) {
    std::lock_guard<std::mutex> g(mailbox_mutex());
    mailbox_cache()[slot]->in_use = false;
}
// a peer's mailbox, mapped once per distinct IPC handle
int peer_map(int device, const cudaIpcMemHandle_t& h, void** base) {
    static std::vector<std::pair<std::string, void*>> maps;
    std::lock_guard<std::mutex> g(mailbox_mutex());
    const std::string key = std::to_string(device) + ":" + std::string(reinterpret_cast<const char*>(&h), sizeof h);
    for (auto& kv : maps) if (kv.first == key) { *base = kv.second; return 0; }
    CU(cudaIpcOpenMemHandle(base, h, cudaIpcMemLazyEnablePeerAccess));
    maps.emplace_back(key, *base);
    return 0;
}
inline ulonglong2* p2p_slots(void* base) { return reinterpret_cast<ulonglong2*>(static_cast<char*>(base) + P2P_HDR_BYTES); }

}  // namespace

extern "C" {

const char* pipsort_last_error(void) { return g_err.c_str(); }
const char* pipsort_version(void) { return "pipsort_b200 0.1 (sm_100a)"; }

void pipsort_destroy(pipsort_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (const pipsort_engine::Alloc& a : e->allocs) a.pinned ? cudaFreeHost(a.p) : cudaFreeAsync(a.p, e->own_stream);
    if (e->arena) cudaFreeAsync(e->arena, e->own_stream);
    if (e->p2p.cache_slot >= 0) mailbox_release(e->p2p.cache_slot);   // mailbox, counters and peer mappings stay with the process
    for (cudaGraphExec_t x : e->graphs) cudaGraphExecDestroy(x);
    if (e->own_stream) kit_release(e->device, StreamKit{e->own_stream, {e->ev0, e->ev1, e->evk0, e->evk1, e->ev_up}, e->pin});
    delete e;
}

// The prior (gamma, p) of log_prior (postcal.cpp:19-59): pi[j][a] = pi'(j,a) = (gamma/(1-gamma))^j p^a ((1-p)/2)^(j-a), the
// complete log prior logprior[j][a] (may be NULL), and *minpi = the smallest finite log pi'(j,a) with j <= kb.  pipsort_create
// (the engine's own prior) and pipsort_read_prior_grid (every prior of a grid) both build their tables here.
static int prior_tables(double gam, double p, int U, int kb, double (*pi)[KMAX + 1], double (*logprior)[KMAX + 1], double* minpi) {
    if (!(gam > 0.0 && gam < 1.0)) return fail(PIPSORT_E_ARG, "gamma must be in (0,1)");
    if (!(p >= 0.0 && p <= 1.0)) return fail(PIPSORT_E_ARG, "sharing_param must be in [0,1]");
    double mn = 0.0;
    for (int j = 0; j <= KMAX; j++)
        for (int a = 0; a <= KMAX; a++) {
            if (a > j) { pi[j][a] = 0.0; if (logprior) logprior[j][a] = 0.0; continue; }
            double lp = 0.0, rel = 0.0;
            if (p != 0.0) {                                   // postcal.cpp:27: the sharing term is skipped for p == 0
                for (int i = 0; i < a; i++) lp += std::log(p);
                for (int i = a; i < j; i++) lp += std::log((1.0 - p) * 0.5);
                rel = lp;
            }
            for (int i = 0; i < j; i++) lp += std::log(gam);
            lp += (U - j) * std::log(1.0 - gam);
            rel += j * (std::log(gam) - std::log(1.0 - gam));
            if (logprior) logprior[j][a] = lp;
            pi[j][a] = std::exp(rel);                         // 0 when p == 1 and a < j
            if (j <= kb && std::isfinite(rel)) mn = std::min(mn, rel);
        }
    if (minpi) *minpi = mn;
    return 0;
}

// log2 of the largest value score_lane.cuh can form under the prior (pi'(k,0) tables, rho = p / ((1-p)/2) finite and
// non-zero), plus 2 LANE_KMAX bits for its sums.  For a row of k SNPs in a warp-step of K >= k SNPs it forms the weights
// w0[j] = pi'(k,0) rho^(j-K) and w1[j] = rho^j (j = 0..K), multiplies them by a table entry (1 for the empty mask, below
// 2^450 for any other) and forms the terms pi'(k,0) rho^a E_0 E_1 (0 <= a <= k) of the expansions.  Its factorised sum
// meets w0[1] E = pi'(k,0) rho^(1-K) E even where every term of the expansions is small: at p = 2e-39 and gamma =
// 0.99999 that is inf for E near 2^450 although rho^8 is a normal double.
static double lane_peak_bits(const double (*pi)[KMAX + 1], double rho) {
    const double lr = std::log2(rho), fast = std::log2(FAST_LIMIT);
    double peak = -INFINITY;
    for (int K = 1; K <= LANE_KMAX; K++)
        for (int k = 1; k <= K; k++) {
            const double lp = std::log2(pi[k][0]);
            for (int j = 0; j <= K; j++) {
                const double e = j > 0 ? fast : 0.0;
                peak = std::max(peak, std::max(lp + (j - K) * lr, j * lr) + e);
            }
            for (int a = 0; a <= k; a++) peak = std::max(peak, lp + a * lr + 2.0 * fast);
        }
    return peak + 2 * LANE_KMAX;
}

// One prior of a grid read as the finalize kernel takes it (PRIOR_STRIDE doubles)
static int grid_prior(const pipsort_engine* e, double gam, double p, double* out) {
    double pi[KMAX + 1][KMAX + 1];
    int rc = prior_tables(gam, p, e->U, e->kb, pi, nullptr, nullptr);
    if (rc) return rc;
    memcpy(out, pi, sizeof pi);
    out[PRIOR_STRIDE - 1] = -0.5 * e->K + e->U * std::log(1.0 - gam);
    return 0;
}

// slot rows of the accumulator store: the five per-SNP slots + the scalars' slot, or (class-resolved) 3 c(c+1)/2 class slots
// per SNP and as many rows as the scalars need (common.cuh)
static size_t store_rows(bool classes, int kb, size_t upad) {
    return classes ? (size_t)cls_nslot(kb) + (cls_nscal(kb) + upad - 1) / upad : (size_t)NSLOT;
}

static int create_impl(const pipsort_locus* lc, int device, uint32_t flags, pipsort_engine* e) {
    const int S = lc->num_studies, U = lc->union_count;
    static const bool trace_create = getenv("PIPSORT_TRACE_CREATE") != nullptr;
    std::chrono::steady_clock::time_point tr[8];
    const auto tr_begin = std::chrono::steady_clock::now();
#define TR(i) do { if (trace_create) tr[i] = std::chrono::steady_clock::now(); } while (0)
    int ndev_now;
    {
        static int ndev = -1;
        std::lock_guard<std::mutex> g(init_mutex());
        if (ndev <= 0 && (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)) {
            ndev = -1;
            return fail(PIPSORT_E_CUDA, "no CUDA device available (the engine has no CPU path)");
        }
        ndev_now = ndev;
    }
    if (device < 0 || device >= ndev_now) return fail(PIPSORT_E_ARG, "device %d out of range (have %d)", device, ndev_now);
    CU(cudaSetDevice(device));
    e->device = device;
    {
        static int sm_cache[64] = {0};
        std::lock_guard<std::mutex> g(init_mutex());
        if (!sm_cache[device & 63]) CU(cudaDeviceGetAttribute(&sm_cache[device & 63], cudaDevAttrMultiProcessorCount, device));
        e->sm_count = sm_cache[device & 63];
    }
    {
        int rcp = pool_setup(device);
        if (rcp) return rcp;
    }
    {
        StreamKit k;
        int rck = kit_acquire(device, &k);
        if (rck) return rck;
        e->own_stream = k.stream; e->ev0 = k.ev[0]; e->ev1 = k.ev[1]; e->evk0 = k.ev[2]; e->evk1 = k.ev[3]; e->ev_up = k.ev[4];
        e->pin = k.pin; e->pin_off = 0;
    }
    e->stream = e->own_stream;
    e->U = U;
    e->K = lc->K; e->gamma = lc->gamma; e->p = lc->sharing_param;
    e->kb = std::min(KMAX, std::max(3, lc->max_causal));
    e->classes = (flags & PIPSORT_PRIOR_CLASSES) != 0;
    e->use_reg_kernel = !(flags & PIPSORT_GENERIC_ONLY);

    TR(0);
    // ---- internal order ---------------------------------------------------------------------------
    std::vector<int> type_user(U);
    for (int g = 0; g < U; g++) {
        const int a = lc->snp_map[g], b = lc->snp_map[U + g];
        if (a >= lc->num_snps[0] || b >= lc->num_snps[1] || a < -1 || b < -1)
            return fail(PIPSORT_E_ARG, "snp_map entry %d out of range", g);
        type_user[g] = (a >= 0 && b >= 0) ? 0 : (a >= 0 ? 1 : (b >= 0 ? 2 : 3));
    }
    e->perm.resize(U);
    for (int g = 0; g < U; g++) e->perm[g] = g;
    if (!(flags & PIPSORT_KEEP_ORDER))
        std::stable_sort(e->perm.begin(), e->perm.end(), [&](int a, int b) { return type_user[a] < type_user[b]; });
    std::vector<int> u2i(U);
    e->types.resize(U);
    for (int i = 0; i < U; i++) { u2i[e->perm[i]] = i; e->types[i] = type_user[e->perm[i]]; }
    e->cost_model = exh_cost_model(U, e->types.data());
    for (int s = 0; s < S; s++) {
        e->n_raw[s] = lc->num_snps[s];
        e->loc[s].assign(U, -1);
        e->orig[s].clear();
        std::vector<char> seen(lc->num_snps[s], 0);
        for (int i = 0; i < U; i++) {
            const int o = lc->snp_map[(size_t)s * U + e->perm[i]];
            if (o < 0) continue;
            if (seen[o]) return fail(PIPSORT_E_ARG, "study %d SNP %d appears twice in the snp_map", s, o);
            seen[o] = 1;
            e->loc[s][i] = (int)e->orig[s].size();
            e->orig[s].push_back(o);
        }
    }

    TR(1);
    // ---- arena: everything dev_alloc hands out below (estimate; the accumulator store is sized for 16 bins) ------------
    {
        const size_t upad = (size_t)std::max((U + 3) & ~3, 4);
        size_t est = 64 * 256 + sizeof(LocusDev) + (size_t)(3 + 5 * U + NCOUNTER) * 8 + (size_t)(U + 2) * 8 +
                     (store_rows(e->classes, e->kb, upad) * 16 * upad + NCOUNTER) * 8;
        est += ((size_t)e->sm_count * 12 + 256) * sizeof(int4) + 512;               // chunk descriptors of the exhaustive launch
        size_t nints = (size_t)6 * U + 2 * ((size_t)U / 32 + 8);
        for (int s = 0; s < S; s++) {
            const size_t nr = (size_t)lc->num_snps[s], n = e->orig[s].size(), ldw = (n + 3) & ~(size_t)3;
            nints += 2 * n + nr;
            est += (7 * nr + n * ldw) * 8;                                        // z upload, six vectors, W
            if (lc->max_causal >= 2 && n <= 4096) est += (n + 1) * (ldw + 4) * 16 + 256;   // WP table (first exhaustive run)
            if (nr * nr * 8 <= ((size_t)4 << 20)) est += nr * nr * 8 + 256;        // small raw LD upload buffer
        }
        est += nints * 4;
        CU(cudaMallocAsync((void**)&e->arena, est, e->own_stream));
        e->arena_cap = est;
        e->arena_off = 0;
    }

    TR(2);
    // ---- device copy of the locus -------------------------------------------------------------------
    LocusDev& L = e->L;
    memset(&L, 0, sizeof L);
    L.U = U;
    int rc;
    // one packed upload of all the small integer arrays:
    //   u2i[U] | snp_map[2U] | loc0[U] | loc1[U] | orig0 | orig1 | raw2loc0 | raw2loc1 | loc2u0 | loc2u1
    int* d_ints = nullptr;
    size_t orig_off[2], r2l_off[2], l2u_off[2], tiles_off = 0;
    std::vector<int> pack;   // function scope: stays alive until the uploads have completed (ev_up below)
    {
        pack.reserve((size_t)5 * U + 2 * (e->orig[0].size() + e->orig[1].size()) + lc->num_snps[0] + lc->num_snps[1]);
        pack.insert(pack.end(), u2i.begin(), u2i.end());
        pack.insert(pack.end(), lc->snp_map, lc->snp_map + (size_t)2 * U);
        for (int s = 0; s < S; s++) pack.insert(pack.end(), e->loc[s].begin(), e->loc[s].end());
        for (int s = 0; s < S; s++) { orig_off[s] = pack.size(); pack.insert(pack.end(), e->orig[s].begin(), e->orig[s].end()); }
        for (int s = 0; s < S; s++) {
            r2l_off[s] = pack.size();
            std::vector<int> r2l(lc->num_snps[s], -1);
            for (size_t l = 0; l < e->orig[s].size(); l++) r2l[e->orig[s][l]] = (int)l;
            pack.insert(pack.end(), r2l.begin(), r2l.end());
        }
        for (int s = 0; s < S; s++) {
            l2u_off[s] = pack.size();
            std::vector<int> l2u(e->orig[s].size(), -1);
            for (int i = 0; i < U; i++) if (e->loc[s][i] >= 0) l2u[e->loc[s][i]] = i;
            pack.insert(pack.end(), l2u.begin(), l2u.end());
        }
        const ExhTiles& tl = e->cost_model.tiles;                      // x tiles of the exhaustive kernel: lo | vmin | of
        tiles_off = pack.size();
        pack.insert(pack.end(), tl.lo.begin(), tl.lo.end());
        pack.insert(pack.end(), tl.vmin.begin(), tl.vmin.end());
        pack.insert(pack.end(), tl.of.begin(), tl.of.end());
        if ((rc = dev_alloc(e, &d_ints, pack.size())) || (rc = upload_small(e, d_ints, pack.data(), pack.size() * sizeof(int)))) return rc;
    }
    L.u2i = d_ints;
    L.ntiles = e->cost_model.tiles.T;
    L.tile_lo = d_ints + tiles_off; L.tile_vmin = L.tile_lo + L.ntiles; L.tile_of = L.tile_vmin + L.ntiles;
    for (int s = 0; s < S; s++) { L.raw2loc[s] = d_ints + r2l_off[s]; L.loc2u[s] = d_ints + l2u_off[s]; L.n_raw[s] = lc->num_snps[s]; }
    e->d_snp_map = d_ints + U;
    size_t soff = 0, zoff = 0;
    double maxexp_nats = 0.0, minexp_bits = 0.0;
    double K_total = (flags & PIPSORT_RAW_LD) ? 0.0 : lc->K;
    TR(3);
    // all host -> device copies of the caller's buffers first, then one event: pipsort_create returns when they are done
    double *up_sigma[2] = {nullptr, nullptr}, *up_z[2] = {nullptr, nullptr};
    DevTemp<double> big_sigma[2];   // a large LD matrix is needed only until the preparation launch has read it
    {
        size_t so = 0, zo = 0;
        for (int s = 0; s < S; s++) {
            const size_t nr = (size_t)lc->num_snps[s];
            if (nr * nr * 8 <= ((size_t)4 << 20)) {          // small: from the arena (stays allocated, a few hundred KB)
                if ((rc = dev_alloc(e, &up_sigma[s], nr * nr))) return rc;
            } else {
                CU(big_sigma[s].alloc(nr * nr, e->stream));
                up_sigma[s] = big_sigma[s];
            }
            CU(cudaMemcpyAsync(up_sigma[s], lc->sigma + so, nr * nr * sizeof(double), cudaMemcpyHostToDevice, e->stream));
            if ((rc = dev_upload(e, &up_z[s], lc->z + zo, nr))) return rc;
            so += nr * nr; zo += nr;
        }
        CU(cudaEventRecord(e->ev_up, e->stream));
    }
    TR(4);
    PrepLocusArgs prep_args;
    memset(&prep_args, 0, sizeof prep_args);
    for (int s = 0; s < S; s++) {
        const int n_raw = lc->num_snps[s], n = (int)e->orig[s].size();
        const int ldw = (n + 3) & ~3;
        const double d = lc->d[s];
        if (!(d > 0.0) || !std::isfinite(d)) return fail(PIPSORT_E_ARG, "d[%d] must be positive and finite", s);
        double *d_sigma = nullptr, *d_zraw = nullptr, *W = nullptr, *A = nullptr, *z = nullptr, *invA = nullptr, *u = nullptr,
               *e1m = nullptr;
        int *d_orig = nullptr, *d_loc = nullptr, *e1n = nullptr;
        d_sigma = up_sigma[s];
        d_zraw = up_z[s];
        if (flags & PIPSORT_RAW_LD) {   // model.h:171-264 on the device: PSD shift + eigen-decomposition -> effective LD, K_s
            std::string why;
            const int prc = prep_study_device(e->stream, n_raw, d_sigma, d_zraw, &e->prep[s], &why, &e->launches);
            if (prc) return fail(prc == -3 ? PIPSORT_E_RANGE : PIPSORT_E_CUDA, "pre-processing of study %d: %s", s, why.c_str());
            K_total += e->prep[s].K;
            e->prepped = true;
        }
        d_orig = d_ints + orig_off[s];
        d_loc = d_ints + (size_t)3 * U + (size_t)s * U;
        if ((rc = dev_alloc(e, &W, (size_t)n * ldw))) return rc;
        if ((rc = dev_alloc(e, &A, n)) || (rc = dev_alloc(e, &z, n)) || (rc = dev_alloc(e, &invA, n)) ||
            (rc = dev_alloc(e, &u, n)) || (rc = dev_alloc(e, &e1m, n)) || (rc = dev_alloc(e, &e1n, n)))
            return rc;
        double2* WP = nullptr;
        const int ldp = (n + 2) & ~1;
        if ((flags & PIPSORT_INTERNAL_WITH_PAIRS) && !(flags & PIPSORT_GENERIC_ONLY) && lc->max_causal >= 2)
            if ((rc = dev_alloc(e, &WP, (size_t)(n + 1) * ldp))) return rc;
        prep_args.s[s] = PrepStudyArgs{d_sigma, d_zraw, d_orig, n_raw, n, ldw, d, W, A, z, invA, u, e1m, e1n, WP, ldp};
        StudyDev& st = L.st[s];
        st.W = W; st.A = A; st.z = z; st.invA = invA; st.u = u; st.e1m = e1m; st.e1n = e1n;
        st.WP = WP; st.ldp = ldp;
        st.n = n; st.ldw = ldw; st.hd = 0.5 * d;
        L.loc[s] = d_loc;
        // exponent range: f_s(C) <= d/2 |z_C|^2 (A >= I), E_s(C) >= prod (1 + d Sigma_ii)^(-1/2)
        std::vector<double> z2;
        double maxdiag = 0.0;
        for (int i = 0; i < n; i++) {
            const int o = e->orig[s][i];
            const double zi = lc->z[zoff + o];
            z2.push_back(zi * zi);
            maxdiag = std::max(maxdiag, std::fabs(lc->sigma[soff + (size_t)o * n_raw + o]) + e->prep[s].add_diag);
        }
        std::sort(z2.begin(), z2.end(), std::greater<double>());
        double top = 0.0;
        for (int i = 0; i < std::min<int>(e->kb, (int)z2.size()); i++) top += z2[i];
        maxexp_nats += 0.5 * d * top;
        minexp_bits -= 0.5 * e->kb * std::log2(1.0 + d * maxdiag);
        soff += (size_t)n_raw * n_raw;
        zoff += n_raw;
    }

    {   // W = d Sigma~ in the internal order + the per-SNP vectors, both studies, one launch
        const bool with_pairs = prep_args.s[0].WP != nullptr;
        const int nmax = std::max(prep_args.s[0].n, prep_args.s[1].n) + (with_pairs ? 1 : 0);
        const int lmax = std::max(std::max(prep_args.s[0].ldw, prep_args.s[1].ldw), with_pairs ? std::max(prep_args.s[0].ldp, prep_args.s[1].ldp) : 0);
        if (nmax > 0) {
            dim3 grid((lmax + 127) / 128, nmax, 2);
            prepare_locus_kernel<<<grid, 128, 0, e->stream>>>(prep_args);
            e->launches++;
            CU(cudaGetLastError());
        }
        for (DevTemp<double>& b : big_sigma) b.free();   // stream-ordered: after the launch that reads it
    }

    TR(5);
    // ---- prior tables (log_prior, postcal.cpp:19-59) --------------------------------------------------
    const double gam = lc->gamma, p = lc->sharing_param;
    double minpi = 0.0;
    if ((rc = prior_tables(gam, p, U, e->kb, L.pi, L.logprior, &minpi))) return rc;
    if (e->classes) minpi = 0.0;     // the class-resolved store holds unweighted sums: the range of the likelihood-only sums
    e->K = K_total;
    L.neg_half_K = -0.5 * K_total;
    L.null_l = (-K_total / 2 - std::sqrt(std::fabs(1.0))) + U * std::log(1.0 - gam);   // postcal.cpp:802-803
    L.cx = -0.5 * K_total + U * std::log(1.0 - gam);
    L.rho = p == 0.0 ? 1.0 : p / ((1.0 - p) * 0.5);
    {
        const double r8 = std::pow(L.rho, KMAX);
        L.lane_ok = p < 1.0 && std::isfinite(r8) && r8 > 0.0 && std::isfinite(1.0 / r8) && lane_peak_bits(L.pi, L.rho) < 1000.0;
    }

    // ---- expansion tables: digit i of e = state of SNP i (0: study 0 only, 1: study 1 only, 2: both) ---
    // locus independent: built once per device and shared by every engine of the process
    {
        static uint32_t* cache[64][KMAX + 1] = {{nullptr}};
        const int dslot = device & 63;
        std::lock_guard<std::mutex> g(init_mutex());      // all KMAX + 1 pointers are published under the lock
        if (!cache[dslot][0]) {
            size_t total = 0;
            int n3s[KMAX + 1];
            for (int k = 0, n3 = 1; k <= KMAX; k++, n3 *= 3) { n3s[k] = n3; total += n3; }
            std::vector<uint32_t> tab(total);
            size_t o = 0;
            for (int k = 0; k <= KMAX; k++)
                for (int x = 0; x < n3s[k]; x++) {
                    uint32_t m0 = 0, m1 = 0, a = 0;
                    int v = x;
                    for (int i = 0; i < k; i++, v /= 3) {
                        const int t = v % 3;
                        if (t != 1) m0 |= 1u << i;
                        if (t != 0) m1 |= 1u << i;
                        if (t == 2) a++;
                    }
                    tab[o++] = m0 | m1 << 8 | a << 16;
                }
            uint32_t* d_tab = nullptr;
            CU(cudaMalloc(&d_tab, total * sizeof(uint32_t)));      // lives as long as the process
            CU(cudaMemcpy(d_tab, tab.data(), total * sizeof(uint32_t), cudaMemcpyHostToDevice));
            o = 0;
            for (int k = 0; k <= KMAX; k++) { cache[dslot][k] = d_tab + o; o += n3s[k]; }
        }
        for (int k = 0; k <= KMAX; k++) L.exptab[k] = cache[dslot][k];
    }

    TR(6);
    // ---- accumulator store ------------------------------------------------------------------------------
    const double maxexp_bits = maxexp_nats * 1.4426950408889634 + 128.0;
    minexp_bits += minpi * 1.4426950408889634 - 128.0;
    if (!(maxexp_bits < 1.0e8) || !(minexp_bits > -1.0e8))
        return fail(PIPSORT_E_RANGE, "exponent range of the locus is out of bounds (z-scores / d too large?)");
    AccDev& acc = L.acc;
    acc.bias = (((int)std::ceil(-minexp_bits) + 511) / 512 + 1) * 512;
    acc.NB = ((int)std::ceil(maxexp_bits) + acc.bias) / 512 + 2;
    acc.Upad = std::max((U + 3) & ~3, 4);
    acc.ccls = e->classes ? e->kb : 0;
    e->bins_len = store_rows(e->classes, e->kb, acc.Upad) * acc.NB * acc.Upad + NCOUNTER;   // the counters ride in the tail of the store
    if ((rc = dev_alloc(e, &acc.bins, e->bins_len))) return rc;
    acc.counters = acc.bins + (e->bins_len - NCOUNTER);
    if ((rc = dev_alloc(e, &e->d_res, 3 + (size_t)5 * U + NCOUNTER))) return rc;   // results | counters: one D2H per read
    e->h_res.resize(3 + (size_t)5 * U + NCOUNTER);
    // scratch of the exhaustive launch (work-queue head, per-a item prefix) from the arena as well
    if ((rc = dev_alloc(e, &e->exh.d_counter, 2))) return rc;
    CU(cudaMemsetAsync(e->exh.d_counter, 0, 2 * sizeof(unsigned), e->stream));
    e->exh.cap_chunks = (size_t)e->sm_count * 12 + 256;     // one chunk per resident warp + singles tiles: the small-locus plan
    if ((rc = dev_alloc(e, &e->exh.d_chunks, e->exh.cap_chunks))) return rc;
    e->exh.pin_stage_cap = e->exh.cap_chunks * sizeof(int4);
    e->exh.pin_stage = pin_slice(e, e->exh.pin_stage_cap);
    CU(cudaMemsetAsync(acc.bins, 0, e->bins_len * sizeof(double), e->stream));
    if (e->classes) {   // the engine's own prior, as the grid finalize reads it (pipsort_finalize must not upload: graphs)
        double own[PRIOR_STRIDE];
        if ((rc = grid_prior(e, gam, p, own))) return rc;
        if ((rc = dev_alloc(e, &e->d_own_prior, PRIOR_STRIDE)) || (rc = upload_small(e, e->d_own_prior, own, sizeof own))) return rc;
    }
    // the caller's buffers and the local staging vectors must not be read after return: wait for the H2D copies only
    // (recorded in ev_up after the last of them); the preparation kernels and memsets keep running asynchronously.
    // e->L lives as long as the engine, so its upload needs no wait.
    e->L_host_copy = e->L;
    if ((rc = dev_alloc(e, &e->d_L, 1)) || (rc = upload_small(e, e->d_L, &e->L_host_copy, sizeof(LocusDev)))) return rc;
    if (!e->defer_upload_sync) CU(cudaEventSynchronize(e->ev_up));
    TR(7);
    if (trace_create) {
        auto us = [&](int a, int b) { return std::chrono::duration<double, std::micro>(tr[b] - tr[a]).count(); };
        fprintf(stderr, "[create] device/kit %.1f | order %.1f | arena %.1f | pack %.1f | uploads %.1f | per-study host %.1f | prep launch+tables %.1f | store+L %.1f us\n",
                std::chrono::duration<double, std::micro>(tr[0] - tr_begin).count(), us(0, 1), us(1, 2), us(2, 3), us(3, 4), us(4, 5), us(5, 6), us(6, 7));
    }
    return 0;
}

int pipsort_create(const pipsort_locus* lc, int device, uint32_t flags, pipsort_engine** out) {
    if (!lc || !out) return fail(PIPSORT_E_ARG, "null argument");
    *out = nullptr;
    if (lc->num_studies != 2)
        return fail(PIPSORT_E_STUDIES, "This prior only works with two studies right now");   // postcal.cpp:20-23
    if (lc->union_count < 0 || !lc->num_snps || !lc->sigma || !lc->z || !lc->d || (!lc->snp_map && lc->union_count))
        return fail(PIPSORT_E_ARG, "incomplete locus description");
    if (lc->num_snps[0] < 0 || lc->num_snps[1] < 0) return fail(PIPSORT_E_ARG, "negative SNP count");
    pipsort_engine* e = new pipsort_engine();
    e->defer_upload_sync = (flags & PIPSORT_INTERNAL_NO_UPLOAD_WAIT) != 0;
    int rc = create_impl(lc, device, flags, e);
    if (rc) { std::string keep = g_err; pipsort_destroy(e); g_err = keep; return rc; }
    *out = e;
    return 0;
}

int pipsort_preprocess_study(int device, int32_t n, const double* ld, const double* z, double* sigma_eff, pipsort_prep_info* info) {
    if (n < 0 || (n > 0 && (!ld || !z || !sigma_eff))) return fail(PIPSORT_E_ARG, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(PIPSORT_E_CUDA, "no CUDA device available (the engine has no CPU path)");
    if (device < 0 || device >= ndev) return fail(PIPSORT_E_ARG, "device %d out of range (have %d)", device, ndev);
    CU(cudaSetDevice(device));
    int rcp = pool_setup(device);
    if (rcp) return rcp;
    cudaStream_t st;
    CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    auto destroy_stream = scope_exit([&] { cudaStreamSynchronize(st); cudaStreamDestroy(st); });   // after the buffers below
    DevTemp<double> dA, dz;
    const size_t nn = (size_t)n * n;
    PrepResult r;
    std::string why;
    unsigned long long launches = 0;
    CU(dA.alloc(nn, st));
    CU(dz.alloc(n, st));
    if (n) CU(cudaMemcpyAsync(dA, ld, nn * sizeof(double), cudaMemcpyHostToDevice, st));
    if (n) CU(cudaMemcpyAsync(dz, z, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
    const int prc = prep_study_device(st, n, dA, dz, &r, &why, &launches);
    if (prc) return fail(prc == -3 ? PIPSORT_E_RANGE : PIPSORT_E_CUDA, "pre-processing: %s", why.c_str());
    if (n) CU(cudaMemcpyAsync(sigma_eff, dA, nn * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (info) { info->add_diag = r.add_diag; info->K = r.K; info->min_abs_eig = r.min_abs_eig; info->n_negative = r.n_negative; info->psd_iterations = r.psd_iterations; }
    return 0;
}

int pipsort_prep_info_get(const pipsort_engine* e, int study, pipsort_prep_info* info) {
    if (!e || !info || study < 0 || study > 1) return fail(PIPSORT_E_ARG, "bad argument");
    if (!e->prepped) return fail(PIPSORT_E_ARG, "the engine was not created with PIPSORT_RAW_LD");
    const PrepResult& r = e->prep[study];
    info->add_diag = r.add_diag; info->K = r.K; info->min_abs_eig = r.min_abs_eig; info->n_negative = r.n_negative; info->psd_iterations = r.psd_iterations;
    return 0;
}

// ---- CUDA graphs: a fixed sequence of the engine's launches (reset + exhaustive + combine + finalize ...) replayed with
// one call -- the launch-bound inner loop of a small locus ------------------------------------------------------------
int pipsort_graph_begin(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (e->capturing) return fail(PIPSORT_E_ARG, "already capturing");
    CU(cudaSetDevice(e->device));
    CU(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
    e->capturing = true;
    return 0;
}

int pipsort_graph_end(pipsort_engine* e, int32_t* graph_id) {
    if (!e || !graph_id) return fail(PIPSORT_E_ARG, "null argument");
    if (!e->capturing) return fail(PIPSORT_E_ARG, "not capturing");
    e->capturing = false;
    cudaGraph_t g = nullptr;
    CU(cudaStreamEndCapture(e->stream, &g));
    cudaGraphExec_t x = nullptr;
    cudaError_t err = cudaGraphInstantiate(&x, g, 0);
    cudaGraphDestroy(g);
    if (err != cudaSuccess) return fail(PIPSORT_E_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(err));
    e->graphs.push_back(x);
    *graph_id = (int32_t)e->graphs.size() - 1;
    return 0;
}

int pipsort_graph_launch(pipsort_engine* e, int32_t graph_id) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (graph_id < 0 || (size_t)graph_id >= e->graphs.size()) return fail(PIPSORT_E_ARG, "unknown graph %d", graph_id);
    CU(cudaGraphLaunch(e->graphs[graph_id], e->stream));
    return 0;
}

int pipsort_reset(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    CU(cudaSetDevice(e->device));
    CU(cudaMemsetAsync(e->L.acc.bins, 0, e->bins_len * sizeof(double), e->stream));
    return 0;
}

int pipsort_total_ranks(const pipsort_engine* e, int c, uint64_t* out) {
    if (!e || !out) return fail(PIPSORT_E_ARG, "null argument");
    if (c < 0) return fail(PIPSORT_E_ARG, "c must be >= 0");
    u64 t = 0;
    bool ovf = false;
    for (int j = 0; j <= std::min(c, e->U); j++) {
        t += binom_host(e->U, j, &ovf);
        if (ovf || t >> 63) return fail(PIPSORT_E_RANGE, "rank space exceeds 2^63 (U=%d, c=%d)", e->U, c);
    }
    *out = t;
    return 0;
}

int pipsort_run_exhaustive(pipsort_engine* e, int c, uint64_t rank_begin, uint64_t rank_end) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (c < 0 || c > e->kb) return fail(PIPSORT_E_ARG, "c=%d outside [0,%d] (max_causal given at create)", c, e->kb);
    uint64_t total = 0;
    int rc = pipsort_total_ranks(e, c, &total);
    if (rc) return rc;
    rank_end = std::min<uint64_t>(rank_end, total);
    if (rank_begin >= rank_end) return 0;
    CU(cudaSetDevice(e->device));
    e->evk_valid = false;
    int jdom = 0;   // the largest subset-size class the range touches: its launch is the dominant kernel
    {
        u64 o = 0;
        for (int j = 0; j <= std::min(c, e->U); j++) {
            const u64 cnt = binom_host(e->U, j, nullptr);
            if (std::max<u64>(rank_begin, o) < std::min<u64>(rank_end, o + cnt)) jdom = j;
            o += cnt;
        }
    }
    // size classes 0..3: one launch of the register kernel (exhaustive.cuh); larger classes: generic kernel
    const int jreg = e->use_reg_kernel ? std::min(std::min(c, 3), e->U) : -1;
    if (jreg >= 2 && !e->L.st[0].WP) {
        // first exhaustive run with pairs / triples: build the tables { W_ij, E_s{i,j} } (16 (n_s + 1)^2 bytes per study, once)
        if (e->capturing) return fail(PIPSORT_E_ARG, "%s", CAPTURE_NO_ALLOC);
        PairTablesArgs pt;
        for (int s = 0; s < 2; s++) {
            StudyDev& st = e->L.st[s];
            double2* WP = nullptr;
            st.ldp = (st.n + 1 + 1) & ~1;
            if ((rc = dev_alloc(e, &WP, (size_t)(st.n + 1) * st.ldp))) return rc;
            st.WP = WP;
            pt.st[s] = st;
            pt.WP[s] = WP;
        }
        const int nmax = std::max(pt.st[0].n, pt.st[1].n), lmax = std::max(pt.st[0].ldp, pt.st[1].ldp);
        {
            dim3 grid((lmax + 127) / 128, nmax + 1, 2);
            pair_tables_kernel<<<grid, 128, 0, e->stream>>>(pt);
            e->launches++;
        }
        CU(cudaGetLastError());
        e->L_host_copy = e->L;
        if ((rc = upload_small(e, e->d_L, &e->L_host_copy, sizeof(LocusDev)))) return rc;
    }
    if (jreg >= 0) {
        const bool timed = jdom <= jreg && !e->capturing;
        if ((rc = exhaustive_plan(e->L, c, rank_begin, rank_end, e->sm_count, &e->exh, &e->cost_model)))
            return fail(PIPSORT_E_CUDA, "exhaustive kernel launch failed: %s", cudaGetErrorString((cudaError_t)rc));
        const size_t nd = e->exh.plan.n_total;     // a larger plan gets headroom: plans differ a little between rank ranges
        if (nd > e->exh.cap_chunks && (rc = grow(e, &e->exh.d_chunks, &e->exh.cap_chunks, nd + nd / 4 + 64))) return rc;
        if ((rc = exhaustive_launch(e->L, e->d_L, e->stream, &e->launches, &e->exh, timed ? e->evk0 : nullptr, timed ? e->evk1 : nullptr)))
            return fail(PIPSORT_E_CUDA, "exhaustive kernel launch failed: %s", cudaGetErrorString((cudaError_t)rc));
        if (timed) e->evk_valid = true;
    }
    u64 off = 0;
    for (int j = 0; j <= std::min(c, e->U); j++) {
        const u64 cnt = binom_host(e->U, j, nullptr);
        const u64 lo = std::max<u64>(rank_begin, off), hi = std::min<u64>(rank_end, off + cnt);
        if (lo < hi && j > jreg) {
            const u64 rb = lo - off, re = hi - off;
            const bool dominant = j == jdom;
            if (dominant && !e->capturing) CU(cudaEventRecord(e->evk0, e->stream));
            size_t smem = 0;
            const int wk = std::max(j, 1);
            if ((rc = ensure_score_smem(e, wk, &smem))) return rc;
            const int chunk = (re - rb) >= (u64)e->sm_count * SCORE_WARPS * 64 ? 16 : 1;
            const u64 nchunks = (re - rb + chunk - 1) / chunk;
            const int blocks = (int)std::min<u64>((nchunks + SCORE_WARPS - 1) / SCORE_WARPS, (u64)e->sm_count * 8);
            if (e->classes) exhaustive_generic_kernel<true><<<blocks, SCORE_WARPS * 32, smem, e->stream>>>(e->L, j, rb, re, chunk, wk);
            else exhaustive_generic_kernel<false><<<blocks, SCORE_WARPS * 32, smem, e->stream>>>(e->L, j, rb, re, chunk, wk);
            e->launches++;
            CU(cudaGetLastError());
            if (dominant && !e->capturing) { CU(cudaEventRecord(e->evk1, e->stream)); e->evk_valid = true; }
        }
        off += cnt;
    }
    return 0;
}

static int check_flags(pipsort_engine* e);
static int flags_to_error(const double* counters);

// mailbox layout: world slots of slot_len 16-byte elements | 8 control words.  A slot = the accumulator store (bins_len
// rounded up to 16) followed by two halves (even / odd rounds) for the shotgun search's per-round exchange: the values of
// up to n_max neighbours + the bins of the running total.
static size_t p2p_acc_len(const pipsort_engine* e) { return (e->bins_len + 15) & ~(size_t)15; }
static size_t p2p_sss_half(const pipsort_engine* e) {
    const size_t n_max = (size_t)e->U * std::max(e->kb, 1) + e->kb + e->U + 1;
    return (n_max + (size_t)e->L.acc.NB + 15) & ~(size_t)15;
}
static size_t p2p_slot_len(const pipsort_engine* e) { return p2p_acc_len(e) + 2 * p2p_sss_half(e); }

// One launch that scores a batch of union configurations: lane per configuration (score_lane.cuh) for up to LANE_KMAX
// SNPs per row, warp per configuration (score.cuh) beyond that, for p == 1 and under PIPSORT_SCORE_WARP=1 (cross-check).
// n_max bounds the batch length for the grid size; the kernel adds *d_n_extra (device) to n when given.
static int launch_score_batch(pipsort_engine* e, const int32_t* d_idx, int64_t n, int64_t n_max, int kmax,
                              const uint8_t* d_make_updates, double* d_out, const int* d_n_extra) {
    static const bool force_warp = getenv("PIPSORT_SCORE_WARP") != nullptr;
    if (kmax <= LANE_KMAX && e->L.lane_ok && !force_warp) {
        if (!e->lane_smem_set) {
            CU(cudaFuncSetAttribute(score_lane_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LANE_SMEM_BYTES));
            e->lane_smem_set = true;
        }
        // the warp-per-configuration fallback inside the kernel needs its shared-memory attribute as well? no: it
        // aliases this kernel's own tables
        const int blocks = (int)std::min<int64_t>((n_max + LANE_CFG_PER_BLOCK - 1) / LANE_CFG_PER_BLOCK, (int64_t)e->sm_count * 8);
        score_lane_kernel<<<std::max(blocks, 1), LANE_THREADS, LANE_SMEM_BYTES, e->stream>>>(e->L, d_idx, n, kmax, d_make_updates,
                                                                                           d_out, d_n_extra);
    } else {
        size_t smem = 0;
        const int wk = std::max(kmax, 1);
        int rc = ensure_score_smem(e, wk, &smem);
        if (rc) return rc;
        const int blocks = (int)std::min<int64_t>((n_max + SCORE_WARPS - 1) / SCORE_WARPS, (int64_t)e->sm_count * 8);
        score_batch_kernel<<<std::max(blocks, 1), SCORE_WARPS * 32, smem, e->stream>>>(e->L, d_idx, n, kmax, wk, d_make_updates, d_out,
                                                                                     d_n_extra);
    }
    e->launches++;
    CU(cudaGetLastError());
    return 0;
}

// what an engine with a class-resolved store (PIPSORT_PRIOR_CLASSES) refuses, and why
static const char* CLASSES_NO_SCORE = "scoring given configurations is not supported on a PIPSORT_PRIOR_CLASSES engine (its store is "
                                      "filled by the exhaustive pass only)";
static const char* CLASSES_NO_SSS = "the shotgun search cannot run on a PIPSORT_PRIOR_CLASSES engine: its search trajectory depends on "
                                    "the prior";

int pipsort_score_union_configs_device(pipsort_engine* e, const int32_t* d_idx, int64_t n, int kmax,
                                       const uint8_t* d_make_updates, double* d_out) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (e->classes) return fail(PIPSORT_E_ARG, "%s", CLASSES_NO_SCORE);
    if (n < 0 || kmax < 0 || kmax > e->kb) return fail(PIPSORT_E_ARG, "kmax=%d outside [0,%d]", kmax, e->kb);
    if (n == 0) return 0;
    CU(cudaSetDevice(e->device));
    return launch_score_batch(e, d_idx, n, n, kmax, d_make_updates, d_out, nullptr);
}

int pipsort_score_union_configs(pipsort_engine* e, const int32_t* idx, int64_t n, int kmax, const uint8_t* make_updates,
                                double* out_max_abs_l) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (e->classes) return fail(PIPSORT_E_ARG, "%s", CLASSES_NO_SCORE);
    if (n < 0 || kmax < 0 || kmax > e->kb) return fail(PIPSORT_E_ARG, "kmax=%d outside [0,%d]", kmax, e->kb);
    if (n == 0) return 0;
    if (!idx && kmax > 0) return fail(PIPSORT_E_ARG, "null idx");
    CU(cudaSetDevice(e->device));
    const size_t ni = (size_t)n * std::max(kmax, 1);
    int rc;
    if ((rc = grow(e, &e->d_idx, &e->cap_idx, ni)) || (rc = grow(e, &e->d_upd, &e->cap_upd, n)) || (rc = grow(e, &e->d_out, &e->cap_out, n)))
        return rc;
    if (kmax > 0) CU(cudaMemcpyAsync(e->d_idx, idx, (size_t)n * kmax * sizeof(int), cudaMemcpyHostToDevice, e->stream));
    if (make_updates) CU(cudaMemcpyAsync(e->d_upd, make_updates, n, cudaMemcpyHostToDevice, e->stream));
    if ((rc = pipsort_score_union_configs_device(e, e->d_idx, n, kmax, make_updates ? e->d_upd : nullptr, e->d_out))) return rc;
    if (out_max_abs_l) CU(cudaMemcpyAsync(out_max_abs_l, e->d_out, n * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    return check_flags(e);      // one synchronisation: the values and the error counters (a refused row, a singular block)
}

int pipsort_score_given_configs_device(pipsort_engine* e, const int16_t* d_configs, int64_t num_configs, int num_groups) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (e->classes) return fail(PIPSORT_E_ARG, "%s", CLASSES_NO_SCORE);
    if (num_configs < 0 || num_groups < 0) return fail(PIPSORT_E_ARG, "negative matrix dimension");
    if (num_configs == 0) return 0;
    if (!d_configs && num_groups > 0) return fail(PIPSORT_E_ARG, "null configs");
    CU(cudaSetDevice(e->device));
    const int64_t blocks = (num_configs + GIVEN_THREADS - 1) / GIVEN_THREADS;
    if (blocks > 0x7fffffff) return fail(PIPSORT_E_ARG, "too many configurations for one call");
    given_configs_kernel<<<(unsigned)blocks, GIVEN_THREADS, 0, e->stream>>>(e->L, d_configs, num_configs, num_groups);
    e->launches++;
    CU(cudaGetLastError());
    return 0;
}

// ---- stochastic shotgun search -----------------------------------------------------------------------------
// first round whose running total is consulted by the convergence rule (sss_postcal.cpp:265-270: "iter >= 100" compares the
// totals after rounds 99 and 100).  The reference's value unless PIPSORT_SSS_CONV_FROM overrides it: a search on a locus
// with a few strong SNPs ends long before round 100, so tests lower the threshold to exercise the rule on such loci (on
// loci with nearly flat likelihoods the search reaches round 100 by itself, tests/search_loci.py).
static int sss_conv_from() {
    const char* v = getenv("PIPSORT_SSS_CONV_FROM");
    return v ? std::max(0, atoi(v)) : 99;
}

static int sss_table_reserve(pipsort_engine* e, u64 need) {   // capacity >= 2 * need
    SssTable& t = e->sss.tab;
    const u64 cap = t.khi ? t.mask + 1 : 0;
    if (cap >= 2 * need && cap) return 0;
    u64 ncap = std::max<u64>(cap, 1u << 16);
    while (ncap < 2 * need) ncap <<= 1;
    SssTable nt{nullptr, nullptr, nullptr, ncap - 1};
    int rc;
    if ((rc = dev_alloc(e, &nt.klo, ncap, Mem::pool)) || (rc = dev_alloc(e, &nt.khi, ncap, Mem::pool)) ||
        (rc = dev_alloc(e, &nt.val, ncap, Mem::pool))) {
        release(e, &nt.klo); release(e, &nt.khi);
        return rc;
    }
    CU(cudaMemsetAsync(nt.khi, 0, ncap * sizeof(u64), e->stream));
    if (t.khi) {
        sss_rehash_kernel<<<(unsigned)((cap + 255) / 256), 256, 0, e->stream>>>(t, nt);
        e->launches++;
        CU(cudaGetLastError());
    }
    SssTable old = t;
    t = nt;
    if ((rc = release(e, &old.klo)) || (rc = release(e, &old.khi)) || (rc = release(e, &old.val))) return rc;
    return 0;
}

int pipsort_sss_reset(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    CU(cudaSetDevice(e->device));
    pipsort_engine::Sss& q = e->sss;
    if (q.tab.khi) CU(cudaMemsetAsync(q.tab.khi, 0, (q.tab.mask + 1) * sizeof(u64), e->stream));
    q.count = 0;
    return 0;
}

// The search on this engine alone (sharded = false) or in lockstep with the ranks of its p2p group, each scoring its share
// of every round's unseen neighbours (sss.cuh).  With one rank no mailbox is touched.
static int sss_run(pipsort_engine* e, int c, int max_iterations, int32_t* iterations, int32_t* stop_reason, bool sharded) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (e->classes) return fail(PIPSORT_E_ARG, "%s", CLASSES_NO_SSS);
    pipsort_engine::P2P& pp = e->p2p;
    if (sharded && !pp.connected) return fail(PIPSORT_E_ARG, "pipsort_p2p_connect has not been called");
    const int U = e->U, world = sharded ? pp.world : 1, rank = sharded ? pp.rank : 0;
    if (c < 0 || c > e->kb) return fail(PIPSORT_E_ARG, "max_causal=%d outside [0,%d] (max_causal given at create)", c, e->kb);
    if (U > SSS_MAX_U) return fail(PIPSORT_E_RANGE, "the search state packs union indices into 15 bits: U=%d > %d", U, SSS_MAX_U);
    if (max_iterations < 0) return fail(PIPSORT_E_ARG, "negative iteration count");
    // at p = 1 every non-empty configuration has an expansion of prior 0, so its largest-|l| value is -inf: the draws
    // would weigh a group by nan (the reference then reads past its neighbourhood list)
    if (c > 0 && e->p == 1.0)
        return fail(PIPSORT_E_ARG, "the shotgun search is undefined at sharing_param = 1 (every neighbour scores -inf)");
    CU(cudaSetDevice(e->device));
    pipsort_engine::Sss& q = e->sss;
    const int kmax = std::max(c, 1);
    const long long n_max = (long long)U * std::max(c, 1) + c + U + 1;
    const size_t m = (size_t)n_max + 1;
    int rc;
    if ((rc = grow(e, &q.d_out_l, &q.cap_out_l, m)) || (rc = grow(e, &q.d_batch, &q.cap_batch, m * kmax)) ||
        (rc = grow(e, &q.d_upd, &q.cap_upd, m)) || (rc = grow(e, &q.d_counter, &q.cap_counter, 2)) ||
        (rc = grow(e, &q.d_scored, &q.cap_scored, m)) || (rc = grow(e, &q.d_state, &q.cap_state, m)) ||
        (rc = grow(e, &q.d_pos_of, &q.cap_pos_of, m)) || (rc = grow(e, &q.d_total, &q.cap_total, 1)) ||
        (rc = grow(e, &q.h_out_l, &q.cap_h_out_l, m + 1, Mem::pinned)) || (rc = pipsort_sss_reset(e)))
        return rc;
    const size_t acc_len = p2p_acc_len(e), half = p2p_sss_half(e), stride = p2p_slot_len(e);
    if (world > 1 && (size_t)n_max + (size_t)e->L.acc.NB > half) return fail(PIPSORT_E_ARG, "mailbox too small for this max_causal");
    double* errf = e->L.acc.counters + 1 + ERR_P2P_TIMEOUT;
    const double cx = -0.5 * e->K + U * std::log(1.0 - e->gamma);     // as finalize_launch: total = log(sum) + cx

    const int conv_from = sss_conv_from();
    std::mt19937 gen(12345);                                             // sss_postcal.cpp:138
    SssCur cur;
    memset(&cur, 0, sizeof cur);                                         // causal_locs starts empty (:115)
    double old_sum_lkl = 0, sss_sum_lkl = 0;
    int iter = 0, why = 0;
    std::vector<double> probs;
    for (iter = 0; iter < max_iterations; iter++) {
        long long nz, nm, np;
        sss_nbd_sizes(U, cur.k, c, nz, nm, np);
        const long long n = nz + nm + np;
        if ((rc = sss_table_reserve(e, q.count + (u64)n))) return rc;
        SssShard sh;
        memset(&sh, 0, sizeof sh);
        sh.world = world; sh.rank = rank;
        if (world > 1) {                                                 // this round's exchange: epoch flag + the half of the slots it uses
            const u64 epoch = ++*pp.sss_epoch;
            sh.flag = (unsigned)(epoch & 0x7fffffffu) + 1u;
            const size_t hoff = acc_len + (size_t)(epoch & 1) * half;
            for (int p = 0; p < world; p++) {
                if (p == rank) continue;
                sh.peer_slot[p] = p2p_slots(pp.peer_base[p]) + (size_t)rank * stride + hoff;
                sh.my_slot[p] = p2p_slots(pp.mailbox) + (size_t)p * stride + hoff;
            }
        }
        CU(cudaMemsetAsync(q.d_counter, 0, 2 * sizeof(int), e->stream));
        sss_lookup_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, e->stream>>>(q.tab, cur, U, c, n, kmax, world, rank, q.d_out_l,
                                                                                 q.d_batch, q.d_upd, q.d_pos_of, q.d_state, q.d_counter);
        e->launches++;
        // one launch scores the current configuration + this rank's unseen neighbours (the batch length is read on the device)
        if ((rc = launch_score_batch(e, q.d_batch, 1, (n + world - 1) / world + 1, kmax, q.d_upd, q.d_scored, q.d_counter))) return rc;
        if (n > 0) {
            if (world > 1) {
                sss_push_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(sh, n, q.d_state, q.d_pos_of, q.d_scored);
                e->launches++;
            }
            sss_insert_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(q.tab, cur, U, c, n, sh, q.d_state, q.d_pos_of,
                                                                                 q.d_scored, q.d_out_l, errf);
            e->launches++;
        }
        if (iter >= conv_from) {                                         // the running sum is only consulted from here on
            sss_total_kernel<<<1, 32, 0, e->stream>>>(e->L.acc, sh, (long long)n_max, cx, q.d_total, errf);
            e->launches++;
        }
        CU(cudaGetLastError());
        int cnt[2] = {0, 0};
        CU(cudaMemcpyAsync(cnt, q.d_counter, sizeof cnt, cudaMemcpyDeviceToHost, e->stream));
        if (n > 0) CU(cudaMemcpyAsync(q.h_out_l, q.d_out_l, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        if (iter >= conv_from) CU(cudaMemcpyAsync(q.h_out_l + n_max + 1, q.d_total, sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        const int n_new = cnt[1];                                        // unseen neighbours of all ranks
        if (n_new == 0) { why = 1; break; }                              // "hit break condition", :260-263
        // (the reference inserts the new values after this check and the next one; the table already holds them, which
        //  is unobservable: both exits leave the loop)
        q.count += (u64)n_new;
        if (iter >= conv_from) sss_sum_lkl = q.h_out_l[n_max + 1];
        if (iter >= conv_from + 1 && (1 - std::exp(old_sum_lkl - sss_sum_lkl)) <= 0.001) { why = 2; break; }   // :265-270

        // sampling, sss_postcal.cpp:289-343: one draw inside each group, then one across the groups
        const double* ll = q.h_out_l;
        double weight[3] = {0.0, 0.0, 0.0};
        long long sample[3] = {n, n, n};
        const long long lo[3] = {0, nz, nz + nm}, hi[3] = {nz, nz + nm, n};
        for (int g = 0; g < 3; g++) {
            if (lo[g] == hi[g]) continue;
            const double max_log = *std::max_element(ll + lo[g], ll + hi[g]);
            probs.clear();
            for (long long ii = lo[g]; ii < hi[g]; ii++) probs.push_back(std::exp(ll[ii] - max_log));
            std::discrete_distribution<size_t> dist(probs.begin(), probs.end());
            sample[g] = (long long)dist(gen);
            weight[g] = std::accumulate(probs.begin(), probs.end(), 0.0);
        }
        std::discrete_distribution<size_t> dist({weight[0], weight[1], weight[2]});
        const size_t grp = dist(gen);
        SssCur nxt;
        memset(&nxt, 0, sizeof nxt);
        nxt.k = sss_neighbour(cur, U, c, sample[grp] + lo[grp], nxt.g);  // :354
        cur = nxt;
        old_sum_lkl = sss_sum_lkl;
    }
    if (iterations) *iterations = iter;
    if (stop_reason) *stop_reason = why;
    return check_flags(e);
}

int pipsort_sss(pipsort_engine* e, int max_causal, int max_iterations, int32_t* iterations, int32_t* stop_reason) {
    return sss_run(e, max_causal, max_iterations, iterations, stop_reason, false);
}

int pipsort_sss_sharded(pipsort_engine* e, int max_causal, int max_iterations, int32_t* iterations, int32_t* stop_reason) {
    return sss_run(e, max_causal, max_iterations, iterations, stop_reason, true);
}

int pipsort_score_given_configs(pipsort_engine* e, const int16_t* configs, int64_t num_configs, int num_groups) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (e->classes) return fail(PIPSORT_E_ARG, "%s", CLASSES_NO_SCORE);
    if (num_configs < 0 || num_groups < 0) return fail(PIPSORT_E_ARG, "negative matrix dimension");
    if (num_configs == 0) return 0;
    if (!configs && num_groups > 0) return fail(PIPSORT_E_ARG, "null configs");
    CU(cudaSetDevice(e->device));
    // stream the matrix through two pinned-size device chunks so that arbitrarily large files (it is mmapped by the
    // caller, postcal.cpp:429) never need more than a bounded staging buffer
    const int64_t rows_per_chunk = std::max<int64_t>(1, ((int64_t)64 << 20) / std::max(1, num_groups * 2));
    DevTemp<int16_t> d_buf[2];
    cudaEvent_t done[2] = {nullptr, nullptr};
    auto destroy_events = scope_exit([&] { for (cudaEvent_t ev : done) if (ev) cudaEventDestroy(ev); });
    const int64_t cap = std::min(rows_per_chunk, num_configs);
    int rc = 0;
    for (int i = 0; i < 2 && !rc; i++) {
        if (d_buf[i].alloc((size_t)cap * std::max(1, num_groups), e->stream) != cudaSuccess ||
            cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) != cudaSuccess)
            rc = fail(PIPSORT_E_CUDA, "staging buffer allocation failed");
        if (num_configs <= cap) break;
    }
    int cur = 0;
    for (int64_t r0 = 0; r0 < num_configs && !rc; r0 += cap, cur ^= 1) {
        const int64_t nr = std::min(cap, num_configs - r0);
        if (r0 >= 2 * cap && cudaEventSynchronize(done[cur]) != cudaSuccess) { rc = fail(PIPSORT_E_CUDA, "event sync failed"); break; }
        if (num_groups > 0 &&
            cudaMemcpyAsync(d_buf[cur], configs + r0 * num_groups, (size_t)nr * num_groups * sizeof(int16_t), cudaMemcpyHostToDevice,
                            e->stream) != cudaSuccess) { rc = fail(PIPSORT_E_CUDA, "H2D copy of the configuration matrix failed"); break; }
        rc = pipsort_score_given_configs_device(e, d_buf[cur], nr, num_groups);
        if (!rc && cudaEventRecord(done[cur], e->stream) != cudaSuccess) rc = fail(PIPSORT_E_CUDA, "event record failed");
    }
    if (rc) return rc;
    return check_flags(e);
}

static int check_flags(pipsort_engine* e) {
    double c[NCOUNTER];
    CU(cudaMemcpyAsync(c, e->L.acc.counters, sizeof c, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return flags_to_error(c);
}

static int flags_to_error(const double* c) {
    if (c[1 + ERR_NOT_PD] != 0.0) return fail(PIPSORT_E_SINGULAR, "matrix is singular");   // postcal.cpp:291-294
    if (c[1 + ERR_RANGE] != 0.0) return fail(PIPSORT_E_RANGE, "a contribution fell outside the provisioned exponent range");
    if (c[1 + ERR_BAD_CONFIG] != 0.0) return fail(PIPSORT_E_CONFIG, "This did not work as expected");   // postcal.cpp:593-596
    if (c[1 + ERR_P2P_TIMEOUT] != 0.0) return fail(PIPSORT_E_CUDA, "a peer did not arrive at the accumulator combine step in time");
    return 0;
}

// the finalize of a class-resolved store for n_priors priors (device table `pri`, PRIOR_STRIDE doubles each) into `res`
static int finalize_grid_launch(pipsort_engine* e, int n_priors, const double* pri, double* res, bool clear) {
    CU(cudaSetDevice(e->device));
    static const bool no_pdl = getenv("PIPSORT_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((e->U + 3 + FIN_WARPS - 1) / FIN_WARPS);
    cfg.blockDim = dim3(FIN_WARPS * 32);
    cfg.stream = e->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = no_pdl ? 0 : 1;
    CU(cudaLaunchKernelEx(&cfg, finalize_grid_kernel, e->L.acc, e->U, n_priors, pri, -0.5 * e->K, res, clear ? 1 : 0));
    e->launches++;
    return 0;
}

static int finalize_launch(pipsort_engine* e, bool clear) {
    // a class-resolved store reports the engine's own prior: the grid finalize for that one prior, same result layout
    if (e->classes) return finalize_grid_launch(e, 1, e->d_own_prior, e->d_res, clear);
    CU(cudaSetDevice(e->device));
    const int U = e->U;
    const double cy = -0.5 * e->K, cx = cy + U * std::log(1.0 - e->gamma);
    static const bool no_pdl = getenv("PIPSORT_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((U + 3 + FIN_WARPS - 1) / FIN_WARPS);
    cfg.blockDim = dim3(FIN_WARPS * 32);
    cfg.stream = e->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = no_pdl ? 0 : 1;
    CU(cudaLaunchKernelEx(&cfg, finalize_kernel, e->L.acc, U, cx, cy, e->d_res, clear ? 1 : 0));
    e->launches++;
    return 0;
}

int pipsort_finalize(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    return finalize_launch(e, false);
}

int pipsort_finalize_reset(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    return finalize_launch(e, true);
}

int pipsort_last_kernel_ms(pipsort_engine* e, float* ms) {
    if (!e || !ms) return fail(PIPSORT_E_ARG, "null argument");
    if (!e->evk_valid) return fail(PIPSORT_E_ARG, "no exhaustive launch recorded");
    CU(cudaSetDevice(e->device));
    CU(cudaEventSynchronize(e->evk1));
    CU(cudaEventElapsedTime(ms, e->evk0, e->evk1));
    return 0;
}

// first half of a read: finalize kernel + device -> host copy of the results, enqueued, not waited for
static int read_enqueue(pipsort_engine* e) {
    int rcf = pipsort_finalize(e);
    if (rcf) return rcf;
    if (!e->h_res_pin) e->h_res_pin = reinterpret_cast<double*>(pin_slice(e, e->h_res.size() * sizeof(double)));
    double* hres = e->h_res_pin ? e->h_res_pin : e->h_res.data();
    CU(cudaMemcpyAsync(hres, e->d_res, e->h_res.size() * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    return 0;
}

static int read_complete(pipsort_engine* e, const pipsort_outputs* out);

int pipsort_fetch_results(pipsort_engine* e, const pipsort_outputs* out) {
    if (!e || !out) return fail(PIPSORT_E_ARG, "null argument");
    CU(cudaSetDevice(e->device));
    if (!e->h_res_pin) e->h_res_pin = reinterpret_cast<double*>(pin_slice(e, e->h_res.size() * sizeof(double)));
    double* hres = e->h_res_pin ? e->h_res_pin : e->h_res.data();
    CU(cudaMemcpyAsync(hres, e->d_res, e->h_res.size() * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    return read_complete(e, out);
}

int pipsort_read_accumulators(pipsort_engine* e, const pipsort_outputs* out) {
    if (!e || !out) return fail(PIPSORT_E_ARG, "null argument");
    int rcf = read_enqueue(e);
    if (rcf) return rcf;
    return read_complete(e, out);
}

static void scatter_results(const pipsort_engine* e, const double* r, const pipsort_outputs* out);

// second half: wait for the engine's stream, check the error counters, scatter into the caller's arrays
static int read_complete(pipsort_engine* e, const pipsort_outputs* out) {
    const int U = e->U;
    double* hres = e->h_res_pin ? e->h_res_pin : e->h_res.data();
    CU(cudaStreamSynchronize(e->stream));
    int rc = flags_to_error(hres + 3 + (size_t)5 * U);
    if (rc) return rc;
    e->last_read_count = (uint64_t)hres[3 + (size_t)5 * U];
    scatter_results(e, hres, out);
    return 0;
}

// results in the finalize kernel's layout (3 + 5 U, internal order) -> the caller's arrays (snp_map / study order)
static void scatter_results(const pipsort_engine* e, const double* r, const pipsort_outputs* out) {
    const int U = e->U;
    if (out->total) *out->total = r[0];
    if (out->noCausal) { out->noCausal[0] = r[1]; out->noCausal[1] = r[2]; }
    r += 3;
    if (out->postValues) {
        const int N = e->n_raw[0] + e->n_raw[1];
        for (int i = 0; i < N; i++) out->postValues[i] = 0.0;
        int offs = 0;
        for (int s = 0; s < 2; s++) {
            for (int g = 0; g < U; g++)
                if (e->loc[s][g] >= 0) out->postValues[offs + e->orig[s][e->loc[s][g]]] = r[(size_t)s * U + g];
            offs += e->n_raw[s];
        }
    }
    for (int g = 0; g < U; g++) {
        const int ug = e->perm[g];
        if (out->sharedPips) out->sharedPips[ug] = r[(size_t)2 * U + g];
        if (out->sharedLL) out->sharedLL[ug] = r[(size_t)3 * U + g];
        if (out->notSharedLL) out->notSharedLL[ug] = r[(size_t)4 * U + g];
    }
}

int pipsort_read_prior_grid(pipsort_engine* e, int n_priors, const double* gamma, const double* sharing_param,
                            const pipsort_outputs* outs, uint64_t* n_configs) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (!e->classes) return fail(PIPSORT_E_ARG, "the engine was not created with PIPSORT_PRIOR_CLASSES: its store holds one prior only");
    if (n_priors < 1) return fail(PIPSORT_E_ARG, "n_priors=%d must be >= 1", n_priors);
    if (!gamma || !sharing_param || !outs) return fail(PIPSORT_E_ARG, "null argument");
    const size_t stride = 3 + (size_t)5 * e->U, npri = (size_t)n_priors * PRIOR_STRIDE;
    const size_t need = npri + (size_t)n_priors * stride + NCOUNTER;
    e->h_grid.resize(need);
    for (int i = 0; i < n_priors; i++) {
        int rc = grid_prior(e, gamma[i], sharing_param[i], e->h_grid.data() + (size_t)i * PRIOR_STRIDE);
        if (rc) { const std::string why = g_err; return fail(rc, "prior %d: %s", i, why.c_str()); }
    }
    CU(cudaSetDevice(e->device));
    int rc;
    if ((rc = grow(e, &e->d_grid, &e->cap_grid, need))) return rc;
    CU(cudaMemcpyAsync(e->d_grid, e->h_grid.data(), npri * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    if ((rc = finalize_grid_launch(e, n_priors, e->d_grid, e->d_grid + npri, false))) return rc;
    CU(cudaMemcpyAsync(e->h_grid.data() + npri, e->d_grid + npri, (need - npri) * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    const double* res = e->h_grid.data() + npri;
    if ((rc = flags_to_error(res + (size_t)n_priors * stride))) return rc;
    e->last_read_count = (uint64_t)res[(size_t)n_priors * stride];
    if (n_configs) *n_configs = e->last_read_count;
    for (int i = 0; i < n_priors; i++) scatter_results(e, res + (size_t)i * stride, &outs[i]);
    return 0;
}

int pipsort_posterior_exhaustive_grid(const pipsort_locus* locus, int device, uint32_t flags, int c, int n_priors, const double* gamma,
                                      const double* sharing_param, const pipsort_outputs* outs, uint64_t* n_configs) {
    if (!outs) return fail(PIPSORT_E_ARG, "null argument");
    if (n_priors < 1) return fail(PIPSORT_E_ARG, "n_priors=%d must be >= 1", n_priors);
    pipsort_engine* e = nullptr;
    int rc = pipsort_create(locus, device, flags | PIPSORT_PRIOR_CLASSES | PIPSORT_INTERNAL_NO_UPLOAD_WAIT |
                                               (c >= 2 ? PIPSORT_INTERNAL_WITH_PAIRS : 0u), &e);
    if (rc) return rc;
    uint64_t total = 0;
    rc = pipsort_total_ranks(e, c, &total);
    if (!rc) rc = pipsort_run_exhaustive(e, c, 0, total);
    if (!rc) rc = pipsort_read_prior_grid(e, n_priors, gamma, sharing_param, outs, n_configs);
    std::string keep = g_err;
    pipsort_destroy(e);
    g_err = keep;
    return rc;
}

int pipsort_posterior_exhaustive(const pipsort_locus* locus, int device, uint32_t flags, int c, const pipsort_outputs* out,
                                 uint64_t* n_configs) {
    if (!out) return fail(PIPSORT_E_ARG, "null argument");
    static const bool trace = getenv("PIPSORT_TRACE") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    const auto t0 = now();
    pipsort_engine* e = nullptr;
    // the caller's buffers stay valid until this function returns: no need to wait for the uploads inside create
    int rc = pipsort_create(locus, device, flags | PIPSORT_INTERNAL_NO_UPLOAD_WAIT | (c >= 2 ? PIPSORT_INTERNAL_WITH_PAIRS : 0u), &e);
    if (rc) return rc;
    const auto t1 = now();
    uint64_t total = 0;
    rc = pipsort_total_ranks(e, c, &total);
    if (!rc) rc = pipsort_run_exhaustive(e, c, 0, total);
    const auto t2 = now();
    if (!rc) rc = pipsort_read_accumulators(e, out);
    const auto t3 = now();
    if (!rc && n_configs) *n_configs = e->last_read_count;
    std::string keep = g_err;
    pipsort_destroy(e);
    g_err = keep;
    if (trace) {
        auto us = [](auto a, auto b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        fprintf(stderr, "[pipsort] create %.1f us, run (enqueue) %.1f us, read (incl. device time) %.1f us, destroy %.1f us\n", us(t0, t1),
                us(t1, t2), us(t2, t3), us(t3, now()));
    }
    return rc;
}

// loci first, first + stride, first + 2 stride, ... through a software pipeline over DEPTH engines, each on its own stream:
// while locus i is being evaluated the uploads and the preparation launches of the next one are already queued, and the
// results of the one DEPTH before are being copied back.  Every locus still pays its own host -> device copy, kernels and
// device -> host read; only the waiting overlaps.  `stop` is raised by the first worker that fails.
static int batch_worker(const pipsort_locus* loci, int32_t n_loci, int first, int stride, int device, uint32_t flags, int c,
                        const pipsort_outputs* outs, uint64_t* n_configs, std::atomic<int>* stop, std::string* err) {
    constexpr int DEPTH = 3;
    pipsort_engine* inflight[DEPTH] = {nullptr, nullptr, nullptr};
    int idx_of[DEPTH] = {-1, -1, -1};
    int rc = 0;
    auto finish = [&](int slot) -> int {       // results of the locus in pipeline slot `slot`
        pipsort_engine*& e = inflight[slot];
        int r = read_complete(e, &outs[idx_of[slot]]);
        if (!r && n_configs) n_configs[idx_of[slot]] = e->last_read_count;
        std::string keep = g_err;
        pipsort_destroy(e);
        g_err = keep;
        e = nullptr;
        return r;
    };
    int k = 0;
    for (int i = first; i < n_loci && !rc && !stop->load(std::memory_order_relaxed); i += stride, k++) {
        const int slot = k % DEPTH;
        if (inflight[slot]) rc = finish(slot);
        if (rc) break;
        pipsort_engine* e = nullptr;
        rc = pipsort_create(&loci[i], device, flags | PIPSORT_INTERNAL_NO_UPLOAD_WAIT | (c >= 2 ? PIPSORT_INTERNAL_WITH_PAIRS : 0u), &e);
        if (rc) break;
        inflight[slot] = e;
        idx_of[slot] = i;
        uint64_t total = 0;
        rc = pipsort_total_ranks(e, c, &total);
        if (!rc) rc = pipsort_run_exhaustive(e, c, 0, total);
        if (!rc) rc = read_enqueue(e);
    }
    // drain in issue order (also after an error: every engine still in flight is destroyed)
    for (int d = 0; d < DEPTH; d++) {
        const int slot = (k + d) % DEPTH;
        if (!inflight[slot]) continue;
        if (!rc && !stop->load(std::memory_order_relaxed)) rc = finish(slot);
        else { std::string keep = g_err; pipsort_destroy(inflight[slot]); g_err = keep; inflight[slot] = nullptr; }
    }
    if (rc) { stop->store(1); *err = g_err; }
    return rc;
}

int pipsort_posterior_exhaustive_batch(const pipsort_locus* loci, int32_t n_loci, int device, uint32_t flags, int c,
                                       const pipsort_outputs* outs, uint64_t* n_configs) {
    if (n_loci < 0 || (n_loci > 0 && (!loci || !outs))) return fail(PIPSORT_E_ARG, "bad argument");
    // The host side of a small locus (a dozen runtime calls, ~60 us) costs as much as its evaluation on the device: long lists
    // are issued by several host threads (PIPSORT_BATCH_THREADS, default 3), each with its own pipeline over its own engines
    // and streams, loci dealt round robin.  The kernels of different loci then also overlap on the device -- a 150-SNP
    // locus is one wave of a latency-bound kernel, and the start-up and the tail of one fill with the steps of another:
    // measured 0.070 / 0.052 / 0.047 ms per locus with 1 / 2 / 3 threads, against 0.053 ms for the kernel alone.
    static const int want = [] { const char* v = getenv("PIPSORT_BATCH_THREADS"); return v ? std::max(1, std::min(8, atoi(v))) : 3; }();
    const int T = n_loci >= 8 ? want : 1;
    std::atomic<int> stop(0);
    std::vector<std::string> errs(T);
    std::vector<int> rcs(T, 0);
    std::vector<std::thread> th;
    for (int t = 1; t < T; t++)
        th.emplace_back([&, t] { rcs[t] = batch_worker(loci, n_loci, t, T, device, flags, c, outs, n_configs, &stop, &errs[t]); });
    rcs[0] = batch_worker(loci, n_loci, 0, T, device, flags, c, outs, n_configs, &stop, &errs[0]);
    for (auto& x : th) x.join();
    for (int t = 0; t < T; t++)
        if (rcs[t]) { g_err = errs[t]; return rcs[t]; }
    return 0;
}

int pipsort_last_read_config_count(const pipsort_engine* e, uint64_t* out) {
    if (!e || !out) return fail(PIPSORT_E_ARG, "null argument");
    *out = e->last_read_count;
    return 0;
}

int pipsort_config_count(pipsort_engine* e, uint64_t* out) {
    if (!e || !out) return fail(PIPSORT_E_ARG, "null argument");
    CU(cudaSetDevice(e->device));
    double c = 0;
    CU(cudaMemcpyAsync(&c, e->L.acc.counters, sizeof c, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    *out = (uint64_t)c;
    return 0;
}

int pipsort_enumerate(pipsort_engine* e, int c, uint64_t rank, uint32_t expansion, int32_t* out_union_idx,
                      int32_t* out_state, uint32_t* n_expansions) {
    if (!e || !out_union_idx || !out_state) return fail(PIPSORT_E_ARG, "null argument");
    if (c < 0 || c > KMAX) return fail(PIPSORT_E_ARG, "c=%d outside [0,%d]", c, KMAX);
    uint64_t total = 0;
    int rc = pipsort_total_ranks(e, c, &total);
    if (rc) return rc;
    if (rank >= total) return fail(PIPSORT_E_ARG, "rank out of range");
    CU(cudaSetDevice(e->device));
    DevTemp<int> d;
    CU(d.alloc(2 * KMAX + 1, e->stream));
    enumerate_kernel<<<1, 32, 0, e->stream>>>(e->U, e->d_snp_map, c, rank, expansion, d, d + KMAX, (unsigned*)(d + 2 * KMAX));
    e->launches++;
    int h[2 * KMAX + 1];
    CU(cudaMemcpyAsync(h, d, sizeof h, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    for (int i = 0; i < c; i++) { out_union_idx[i] = h[i]; out_state[i] = h[KMAX + i]; }
    if (n_expansions) *n_expansions = (uint32_t)h[2 * KMAX];
    return 0;
}

int pipsort_accumulator_buffer(pipsort_engine* e, void** device_ptr, uint64_t* num_doubles) {
    if (!e || !device_ptr || !num_doubles) return fail(PIPSORT_E_ARG, "null argument");
    *device_ptr = e->L.acc.bins;
    *num_doubles = e->bins_len;
    return 0;
}

int pipsort_merge(pipsort_engine* dst, pipsort_engine* src) {
    if (!dst || !src) return fail(PIPSORT_E_ARG, "null engine");
    if (dst->bins_len != src->bins_len || dst->L.acc.bias != src->L.acc.bias || dst->U != src->U)
        return fail(PIPSORT_E_ARG, "engines were not created from the same locus");
    CU(cudaSetDevice(src->device));
    CU(cudaStreamSynchronize(src->stream));
    CU(cudaSetDevice(dst->device));
    DevTemp<double> tmp;
    const double* from = src->L.acc.bins;
    if (src->device != dst->device) {
        CU(tmp.alloc(dst->bins_len, dst->stream));
        CU(cudaMemcpyPeerAsync(tmp, dst->device, src->L.acc.bins, src->device, dst->bins_len * sizeof(double), dst->stream));
        from = tmp;
    }
    add_bins_kernel<<<(unsigned)((dst->bins_len + 255) / 256), 256, 0, dst->stream>>>(dst->L.acc.bins, from, dst->bins_len);
    dst->launches++;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(dst->stream));
    return 0;   // the configuration count and the error counters are part of the store
}

static int shard_by_types(const std::vector<int>& types, int c, int parts, uint64_t* bounds);

// ---- peer-memory combine -----------------------------------------------------------------------------------


int pipsort_p2p_export(pipsort_engine* e, int world, void* handle) {
    if (!e || !handle) return fail(PIPSORT_E_ARG, "null argument");
    if (world < 1 || world > P2P_MAX_WORLD) return fail(PIPSORT_E_ARG, "world=%d outside [1,%d]", world, P2P_MAX_WORLD);
    CU(cudaSetDevice(e->device));
    pipsort_engine::P2P& q = e->p2p;
    if (q.mailbox && q.world != world) return fail(PIPSORT_E_ARG, "mailbox already exported for world=%d", q.world);
    if (!q.mailbox) {
        const size_t bytes = P2P_HDR_BYTES + (size_t)world * p2p_slot_len(e) * sizeof(ulonglong2);
        int rc = mailbox_acquire(e->device, world, bytes, &q.cache_slot);
        if (rc) return rc;
        MailboxEntry* m = mailbox_cache()[q.cache_slot];
        q.mailbox = m->mailbox;
        q.d_done = m->d_done;
        q.sss_epoch = &m->sss_epoch;
        q.world = world;
    }
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, q.mailbox));
    static_assert(sizeof(cudaIpcMemHandle_t) == PIPSORT_IPC_HANDLE_BYTES, "IPC handle size");
    memcpy(handle, &h, sizeof h);
    return 0;
}

int pipsort_p2p_connect(pipsort_engine* e, const void* handles, int world, int rank, int root) {
    if (!e || !handles) return fail(PIPSORT_E_ARG, "null argument");
    if (world < 1 || world > P2P_MAX_WORLD || rank < 0 || rank >= world || root < 0 || root >= world)
        return fail(PIPSORT_E_ARG, "bad world/rank/root (%d/%d/%d)", world, rank, root);
    pipsort_engine::P2P& q = e->p2p;
    if (!q.mailbox || q.world != world) return fail(PIPSORT_E_ARG, "call pipsort_p2p_export with the same world first");
    if (q.connected) return fail(PIPSORT_E_ARG, "already connected");
    CU(cudaSetDevice(e->device));
    q.rank = rank; q.root = root;
    q.peers.world = world; q.peers.root = root;
    for (int r = 0; r < world; r++) {
        void* base = q.mailbox;
        if (r != rank) {
            cudaIpcMemHandle_t h;
            memcpy(&h, (const char*)handles + (size_t)r * PIPSORT_IPC_HANDLE_BYTES, sizeof h);
            int rc = peer_map(e->device, h, &base);
            if (rc) return rc;
        }
        q.peer_base[r] = base;
        q.peers.ctrl[r] = reinterpret_cast<u64*>(base);          // the control words open the mailbox
    }
    q.connected = true;
    return 0;
}

static int p2p_reduce_impl(pipsort_engine* e, bool clear_sender);
int pipsort_p2p_reduce_to_root(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    return p2p_reduce_impl(e, false);
}
int pipsort_p2p_reduce_to_root_reset(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    return p2p_reduce_impl(e, true);
}
static int finalize_launch(pipsort_engine* e, bool clear);
int pipsort_p2p_combine_finalize(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    if (e->classes)
        return fail(PIPSORT_E_ARG, "the fused combine + finalize reads the five-slot store only; on a PIPSORT_PRIOR_CLASSES engine "
                                   "use pipsort_p2p_reduce_to_root and read the root");
    pipsort_engine::P2P& q = e->p2p;
    if (!q.connected) return fail(PIPSORT_E_ARG, "pipsort_p2p_connect has not been called");
    if (q.world == 1) return finalize_launch(e, true);
    if (q.rank != q.root) return p2p_reduce_impl(e, true);
    if (e->L.acc.NB > 32) {                          // many bins: merge into the store, then the scanning finalize
        int rc = p2p_reduce_impl(e, true);
        return rc ? rc : finalize_launch(e, true);
    }
    CU(cudaSetDevice(e->device));
    const int U = e->U;
    const double cy = -0.5 * e->K, cx = cy + U * std::log(1.0 - e->gamma);
    static const bool no_pdl = getenv("PIPSORT_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((U + 3 + FIN_WARPS - 1) / FIN_WARPS);
    cfg.blockDim = dim3(FIN_WARPS * 32);
    cfg.stream = e->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = no_pdl ? 0 : 1;
    double* errf = e->L.acc.counters + 1 + ERR_P2P_TIMEOUT;
    CU(cudaLaunchKernelEx(&cfg, finalize_merge_kernel, e->L.acc, U, cx, cy, e->d_res, p2p_slots(q.mailbox),
                          p2p_slot_len(e), e->bins_len, q.peers.ctrl[q.rank], q.peers, q.rank, q.d_done, errf));
    e->launches++;
    return 0;
}

static int p2p_reduce_impl(pipsort_engine* e, bool clear_sender) {
    pipsort_engine::P2P& q = e->p2p;
    if (!q.connected) return fail(PIPSORT_E_ARG, "pipsort_p2p_connect has not been called");
    if (q.world == 1) return 0;
    CU(cudaSetDevice(e->device));
    const size_t n = e->bins_len, slot = p2p_slot_len(e);
    const unsigned blocks = (unsigned)std::min<size_t>((n + 511) / 512, (size_t)e->sm_count * 2);
    double* errf = e->L.acc.counters + 1 + ERR_P2P_TIMEOUT;
    static const bool no_pdl = getenv("PIPSORT_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(blocks);
    cfg.blockDim = dim3(256);
    cfg.stream = e->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = no_pdl ? 0 : 1;
    if (q.rank != q.root) {
        CU(cudaLaunchKernelEx(&cfg, p2p_push_kernel, e->L.acc.bins, n, p2p_slots(q.peer_base[q.root]) + (size_t)q.rank * slot,
                              q.peers.ctrl[q.rank], q.d_done, errf, clear_sender ? 1 : 0));
    } else {
        CU(cudaLaunchKernelEx(&cfg, p2p_merge_kernel, e->L.acc.bins, (const ulonglong2*)p2p_slots(q.mailbox), n, slot,
                              q.peers.ctrl[q.rank], q.peers, q.rank, q.d_done, errf));
    }
    e->launches++;
    return 0;
}

int pipsort_shard_ranks(const pipsort_engine* e, int c, int parts, uint64_t* bounds) {
    if (!e || !bounds || parts < 1) return fail(PIPSORT_E_ARG, "bad argument");
    return shard_by_types(e->types, c, parts, bounds);
}

int pipsort_shard_ranks_for_map(const int32_t* snp_map, int32_t union_count, int c, int parts, uint32_t flags, uint64_t* bounds) {
    if ((!snp_map && union_count) || union_count < 0 || !bounds || parts < 1) return fail(PIPSORT_E_ARG, "bad argument");
    const int U = union_count;
    std::vector<int> types(U);
    for (int g = 0; g < U; g++) {
        const int a = snp_map[g], b = snp_map[U + g];
        types[g] = (a >= 0 && b >= 0) ? 0 : (a >= 0 ? 1 : (b >= 0 ? 2 : 3));
    }
    if (!(flags & PIPSORT_KEEP_ORDER)) std::stable_sort(types.begin(), types.end());   // the engine's internal relabelling
    return shard_by_types(types, c, parts, bounds);
}

static int shard_by_types(const std::vector<int>& types, int c, int parts, uint64_t* bounds) {
    if (c < 0) return fail(PIPSORT_E_ARG, "c must be >= 0");
    const int U = (int)types.size(), cc = std::min(c, U);
    uint64_t total = 0;
    {
        bool ovf = false;
        for (int j = 0; j <= cc; j++) {
            total += binom_host(U, j, &ovf);
            if (ovf || total >> 63) return fail(PIPSORT_E_RANGE, "rank space exceeds 2^63 (U=%d, c=%d)", U, c);
        }
    }
    WorkModel wm(types, std::max(cc, 1));
    // Cost model.  Size classes 2 and 3 run in the register kernel, whose unit of work is a WARP-STEP (a, b, 32-wide
    // tile of x); what a step costs depends on which specialised loop its segment runs (ExhCostModel restates the kernel's
    // dispatch: generic / single-study tile with or without a bordered-step chain).  A segment of ranks is weighted by the
    // cost of its warp-steps, not by its expanded configurations.  Larger classes (generic kernel, one warp per subset) are
    // weighted per subset.
    const ExhCostModel M = exh_cost_model(U, types.data());
    auto tcost = [&](int J, int a, int b) -> double {          // cost of the warp-steps (a, b, all tiles of x > b)
        if (b + 1 >= U) return 0.0;
        return M.tiles_cost(J, a, b, 1, M.tiles.first_tile(b));
    };
    std::vector<double> w3(U + 1, 0.0);           // w3[a] = sum over b > a
    for (int a = U - 2; a >= 0; a--)
        for (int b = a + 1; b + 1 < U; b++) w3[a] += tcost(3, a, b);
    // segments of consecutive ranks (size class j, smallest element g) with their work estimate
    struct Seg { u64 begin, count; double work; };
    std::vector<Seg> segs;
    u64 off = 0;
    for (int j = 0; j <= cc; j++) {
        if (j == 0) { segs.push_back({off, 1, 0.01}); off += 1; continue; }
        for (int g = 0; g + j <= U; g++) {
            const u64 cnt = binom_host(U - 1 - g, j - 1, nullptr);
            double work;
            if (j == 1) work = 1.0 / 32.0;
            else if (j == 2) work = tcost(2, -1, g);
            else if (j == 3) work = w3[g];
            else work = (0.3 * wm.configs_first(j, g) / std::max(1.0, wm.w[g]) + 3.0 * (double)cnt);   // generic kernel: per subset
            segs.push_back({off, cnt, work});
            off += cnt;
        }
    }
    double tw = 0.0;
    for (const Seg& s : segs) tw += s.work;
    bounds[0] = 0;
    bounds[parts] = total;
    size_t si = 0;
    double acc = 0.0;
    for (int p = 1; p < parts; p++) {
        const double target = tw * p / parts;
        while (si < segs.size() && acc + segs[si].work < target) acc += segs[si++].work;
        u64 b = total;
        if (si < segs.size()) {
            const double frac = segs[si].work > 0 ? (target - acc) / segs[si].work : 0.0;
            b = segs[si].begin + (u64)(frac * (double)segs[si].count);
        }
        bounds[p] = std::max<uint64_t>(bounds[p - 1], std::min<uint64_t>(b, total));
    }
    return 0;
}

void* pipsort_stream(pipsort_engine* e) { return e ? (void*)e->stream : nullptr; }

int pipsort_set_stream(pipsort_engine* e, void* cuda_stream) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    CU(cudaSetDevice(e->device));
    CU(cudaStreamSynchronize(e->stream));
    e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
    return 0;
}

int pipsort_flush_l2(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    CU(cudaSetDevice(e->device));
    const size_t bytes = (size_t)256 << 20;   // L2 is 126 MB
    int rc = grow(e, &e->l2_scratch, &e->cap_l2, bytes);
    if (rc) return rc;
    CU(cudaMemsetAsync(e->l2_scratch, 0x5a, bytes, e->stream));
    return 0;
}

int pipsort_sync(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    CU(cudaSetDevice(e->device));
    CU(cudaStreamSynchronize(e->stream));
    return 0;
}

int pipsort_timer_begin(pipsort_engine* e) {
    if (!e) return fail(PIPSORT_E_ARG, "null engine");
    CU(cudaSetDevice(e->device));
    CU(cudaEventRecord(e->ev0, e->stream));
    return 0;
}

int pipsort_timer_end(pipsort_engine* e, float* ms) {
    if (!e || !ms) return fail(PIPSORT_E_ARG, "null argument");
    CU(cudaSetDevice(e->device));
    CU(cudaEventRecord(e->ev1, e->stream));
    CU(cudaEventSynchronize(e->ev1));
    CU(cudaEventElapsedTime(ms, e->ev0, e->ev1));
    return 0;
}

uint64_t pipsort_launch_count(const pipsort_engine* e) { return e ? e->launches : 0; }

int pipsort_measure_fp64_peak(int device, double* flops_per_sec) {
    if (!flops_per_sec) return fail(PIPSORT_E_ARG, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(PIPSORT_E_CUDA, "no CUDA device available");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    DevTemp<double> d;
    CU(d.alloc(1, 0));
    cudaEvent_t a = nullptr, b = nullptr;
    auto destroy_events = scope_exit([&] { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); });
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {
        CU(cudaEventRecord(a));
        dfma_peak_kernel<<<blocks, threads>>>(d, iters, 0.999999, 1.0e-7);
        CU(cudaEventRecord(b));
        CU(cudaEventSynchronize(b));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, a, b));
        const double fl = 2.0 * 64.0 * iters * (double)blocks * threads;
        if (rep > 0) best = std::max(best, fl / (ms * 1e-3));
    }
    *flops_per_sec = best;
    return 0;
}

}  // extern "C"
