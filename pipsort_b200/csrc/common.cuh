// Device-side description of a locus and of the accumulator store, as laid out in HBM by
// pipsort_create (engine.cu).  See DESIGN.md for the derivation; reference citations are relative to
// the PIPSORT source tree.
//
// Closed form (SURVEY.md section 0, restating lowrank_likelihood, postcal.cpp:214-304):
//     just_ll(C0,C1) = -K/2 + f_0(C0) + f_1(C1),   f_s(C) = d_s/2 z_C^T A^-1 z_C - 1/2 log det A,
//     A = I + d_s Sigma~_s[C,C]  (SPD, A >= I).
// The engine works with  E_s(C) = exp(f_s(C))  carried as  m * 2^n  (xacc.cuh) and accumulates
//     X-type sums  sum pi'(j,a) E_0 E_1      (prior-weighted: total, noCausal, postValues, sharedPips)
//     Y-type sums  sum         E_0 E_1      (likelihood only: sharedLL, notSharedLL)
// where pi'(j,a) = (gamma/(1-gamma))^j p^a ((1-p)/2)^(j-a)  is log_prior (postcal.cpp:19-59) without its
// configuration-independent part U log(1-gamma); that part and -K/2 are added back when the logs are
// taken (finalize kernel).
//
// Internal SNP order.  All sums are order independent, so unless PIPSORT_KEEP_ORDER is given the union
// SNPs are relabelled by TYPE (present in both studies / study 0 only / study 1 only) and each study's
// LD and z are permuted into the order of appearance in that relabelled union list.  Consecutive
// internal union SNPs then have consecutive study-local indices (coalesced LD rows) and the same
// number of states (uniform control flow inside a warp).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "xacc.cuh"

namespace pipsort {

constexpr int KMAX = 8;      // PIPSORT_KMAX
constexpr int NSTUDY = 2;    // postcal.cpp:20-23

struct StudyDev {
    const double* W;     // d_s * Sigma~_s, n x ldw row-major, internal local order    (tmp_CC - I, postcal.cpp:276)
    const double* A;     // 1 + W[i][i]
    const double* z;     // B_s^T S'_s
    const double* invA;  // 1 / A[i]
    const double* u;     // z[i] / A[i]
    const double* e1m;   // E_s({i}) = exp(hd z^2/A) / sqrt(A) = e1m * 2^e1n
    const int* e1n;
    const double2* WP;   // LD + pair table of the exhaustive kernel, (n + 1) x ldp: WP[i][j] = { W[i][j], E_s({i,j}) as a plain
                         // double, +inf when it leaves the fast range }; row n and column n are all zero (an absent SNP reads
                         // W = 0, E = 0 without a predicate).  Built on the first exhaustive run with c >= 2; nullptr before.
    int ldp;             // row length of WP (>= n + 1)
    int n;               // SNPs of this study that appear in the snp_map
    int ldw;
    double hd;           // d_s / 2
};

// Per-SNP accumulator slots:
//   X1: prior-weighted sum over configurations where the SNP is causal in study 0 only
//   X2: ... in study 1 only        X3: ... in both studies
//   YS: likelihood-only sum where causal in both,  YN: where causal in exactly one study
// postValues(study 0) = X1+X3, postValues(study 1) = X2+X3, sharedPips = X3, sharedLL = YS,
// notSharedLL = YN   (postcal.cpp:1003-1030)
enum Slot : int { X1 = 0, X2 = 1, X3 = 2, YS = 3, YN = 4, SCAL = 5, NSLOT = 6 };
// slot SCAL holds the scalars at SNP index 0..2
enum Scalar : int { S_TOTAL = 0, S_NC0 = 1, S_NC1 = 2 };

// Accumulator store: every accumulator is a row of NB plain doubles ("bins"); bin b holds the partial
// sum of all contributions whose binary exponent lies in [512 b - bias, 512 b - bias + 512), scaled by
// 2^-(512 b - bias).  A contribution is therefore ONE native fp64 atomic add (RED.E.ADD.F64), needs no
// re-basing, and the store of several GPUs is combined by an element-wise sum (one NCCL all-reduce).
// Layout: bins[(slot * NB + b) * Upad + g].
struct AccDev {
    double* bins;
    int NB;
    int bias;
    int Upad;
    int ccls;          // 0: the store above;  C > 0: the class-resolved store of PIPSORT_PRIOR_CLASSES for size classes <= C (below)
    double* counters;  // tail of the same allocation as bins: [0] expanded configurations evaluated (the reference's
                       // mycount; exact below 2^53), [1 + f] number of times error f was raised.  Doubles, so that the
                       // ONE all-reduce(sum) that combines the stores of several GPUs carries them as well.
};
enum ErrFlag : int { ERR_RANGE = 0, ERR_NOT_PD = 1, ERR_BAD_CONFIG = 2, ERR_P2P_TIMEOUT = 3, NERRFLAG = 4 };
constexpr int NCOUNTER = 1 + NERRFLAG;

struct LocusDev {
    StudyDev st[NSTUDY];
    int U;
    const int* loc[NSTUDY];   // [U] internal union index -> study-local index or -1
    const int* u2i;           // [U] snp_map (user) union index -> internal union index
    const int* raw2loc[NSTUDY];  // [n_raw] study index as in the LD / z files -> study-local internal index or -1
    const int* loc2u[NSTUDY];    // [n] study-local internal index -> internal union index
    int n_raw[NSTUDY];           // PostCal::num_snps_all
    double pi[KMAX + 1][KMAX + 1];        // pi'(j,a)
    double logprior[KMAX + 1][KMAX + 1];  // log_prior(j,a), complete (postcal.cpp:19-59)
    double neg_half_K;                    // -K/2
    double null_l;                        // -K/2 - 1 + U log(1-gamma)   (postcal.cpp:797-803)
    double cx;                            // -K/2 + U log(1-gamma): what the prior-weighted sums leave out
    double rho;                           // pi'(j, a+1) / pi'(j, a) = p / ((1-p)/2)   (1 when p == 0: postcal.cpp:27)
    int lane_ok;                          // the prior factorises with a finite rho (p < 1) and every value score_lane.cuh
                                          // forms fits a double (engine.cu lane_peak_bits): that kernel may be used
    const uint32_t* exptab[KMAX + 1];     // exptab[k][e] = m0 | m1 << 8 | a << 16 for expansion e of a k-subset
    // x tiles of the exhaustive kernel (exh_plan.h, ExhTiles): lane l of tile t is x = tile_lo[t] + l, valid when
    // x >= tile_vmin[t]; tile_of[x] = the tile of x.  Tiles never straddle a boundary between SNP types.
    const int* tile_lo;
    const int* tile_vmin;
    const int* tile_of;
    int ntiles;
    AccDev acc;
};

__device__ __forceinline__ void count_add(const AccDev& a, unsigned long long n) { atomicAdd(a.counters, (double)n); }
__device__ __forceinline__ void flag_set(const AccDev& a, ErrFlag f) {
    if (*(volatile double*)(a.counters + 1 + f) == 0.0) atomicAdd(a.counters + 1 + f, 1.0);   // rare: error path
}

__device__ __forceinline__ double* bin_ptr(const AccDev& a, int slot, int g) {
    return a.bins + (size_t)slot * a.NB * a.Upad + g;
}

// acc[slot][g] += M * 2^N   (M >= 0)
__device__ __forceinline__ void bin_add(const AccDev& a, int slot, int g, double M, int N) {
    if (!(M > 0.0)) return;
    if (M < 1.0e-200) { M *= 0x1p+700; N -= 700; }   // possibly subnormal: make it normal first
    int hi = __double2hiint(M);
    int e = ((hi >> 20) & 0x7ff) - 1023;
    M = __hiloint2double(hi - (e << 20), __double2loint(M));   // mantissa in [1,2)
    int t = N + e + a.bias;
    int b = t >> 9;
    if (b < 0 || b >= a.NB) { flag_set(a, ERR_RANGE); return; }
    atomicAdd(bin_ptr(a, slot, g) + (size_t)b * a.Upad, M * pow2c(t & 511));
}

__device__ __forceinline__ void bin_add(const AccDev& a, int slot, int g, const XAcc& v) { bin_add(a, slot, g, v.M, v.N); }

// The accumulator whose top non-empty bin is `top`, as M * 2^N with M in [1,2): that bin plus the two below it, each scaled
// down by 2^512 per bin (what lies in lower bins is below one ulp of the sum).  bin(k) returns bin top - k; it is called
// only for bins that exist, so that a reader from memory loads no more than it needs.
template <class Bin>
__device__ __forceinline__ XAcc bins_decode(int top, int bias, Bin bin) {
    double M = bin(0);
    if (top > 0) M += bin(1) * 0x1p-512;
    if (top > 1) M += (bin(2) * 0x1p-512) * 0x1p-512;
    const int hi = __double2hiint(M);
    const int e = ((hi >> 20) & 0x7ff) - 1023;
    M = __hiloint2double(hi - (e << 20), __double2loint(M));
    return XAcc{M, 512 * top - bias + e};
}

// Class-resolved store (PIPSORT_PRIOR_CLASSES, DESIGN.md section 5f): the same bins, but every accumulator is UNWEIGHTED and
// resolved by prior class, so that any prior (gamma, p) can be applied when the results are read.
//   per SNP g: G[g][J][t][a'] for J = 1..C, t = 0 / 1 / 2 (study 0 only / study 1 only / both), a' = 0..J-1 other SNPs of
//              the subset causal in both studies -- slot cls_slot(J, t, a');
//   scalars:   T[J][a] (J = 0..C, a = 0..J: every expanded configuration), N_0[J] / N_1[J] (study 0 / study 1 carries no
//              causal SNP, the terms of S_NC0 / S_NC1) -- scalar k lives in slot cls_nslot(C) + k / Upad at column k % Upad.
__host__ __device__ constexpr int cls_slot(int J, int t, int ap) { return 3 * J * (J - 1) / 2 + t * J + ap; }
__host__ __device__ constexpr int cls_nslot(int C) { return 3 * C * (C + 1) / 2; }
__host__ __device__ constexpr int cls_T(int J, int a) { return J * (J + 1) / 2 + a; }
__host__ __device__ constexpr int cls_ntab(int C) { return (C + 1) * (C + 2) / 2; }   // classes (J, a) with J <= C
__host__ __device__ constexpr int cls_N(int C, int s, int J) { return cls_ntab(C) + s * (C + 1) + J; }
__host__ __device__ constexpr int cls_nscal(int C) { return cls_ntab(C) + 2 * (C + 1); }

// Count table (PIPSORT_CAUSAL_COUNTS, DESIGN.md section 5f): a class-resolved store that also keeps R[a][b0][b1], the total
// split by a SNPs causal in both studies, b0 in study 0 only and b1 in study 1 only (J = a + b0 + b1 <= C), as the scalars
// after cls_nscal(C).  Within size class J the classes follow a, then b0; the table at any c is the prefix of the one at C.
__host__ __device__ constexpr int cnt_idx(int J, int a, int b0) { return J * (J + 1) * (J + 2) / 6 + a * (2 * J + 3 - a) / 2 + b0; }
__host__ __device__ constexpr int cnt_ntab(int C) { return (C + 1) * (C + 2) * (C + 3) / 6; }   // classes (a, b0, b1) with J <= C
__host__ __device__ constexpr int cls_R(int C, int J, int a, int b0) { return cls_nscal(C) + cnt_idx(J, a, b0); }

// What the accumulator store holds, and so which instantiation of the exhaustive kernels an engine launches: the five-slot
// store of one prior, the class-resolved store (PIPSORT_PRIOR_CLASSES), or that store with the count table (PIPSORT_CAUSAL_COUNTS)
enum StoreKind : int { STORE_PLAIN = 0, STORE_CLASSES = 1, STORE_COUNTS = 2 };

// scalar k of the class-resolved store += M * 2^N
__device__ __forceinline__ void scal_add(const AccDev& a, int k, double M, int N) {
    bin_add(a, cls_nslot(a.ccls) + k / a.Upad, k % a.Upad, M, N);
}

// Call-local device memory: allocated from the device's pool on `stream`, freed on the same stream when it leaves scope, on
// every return path.
template <class T>
struct DevTemp {
    T* p = nullptr;
    cudaStream_t stream = nullptr;
    DevTemp() = default;
    DevTemp(const DevTemp&) = delete;   // one owner: freed once
    void operator=(const DevTemp&) = delete;
    ~DevTemp() { free(); }
    void free() { if (p) cudaFreeAsync(p, stream); p = nullptr; }   // before scope exit: the memory is not needed any more
    operator T*() const { return p; }
    cudaError_t alloc(size_t count, cudaStream_t s) {
        stream = s;
        const cudaError_t err = cudaMallocAsync((void**)&p, (count ? count : 1) * sizeof(T), s);
        if (err != cudaSuccess) { p = nullptr; cudaGetLastError(); }   // a refused request leaves no error pending
        return err;
    }
};

// Runs f when it leaves scope (handles and events of a call, released on every return path)
template <class F>
struct ScopeExit {
    F f;
    ~ScopeExit() { f(); }
};
template <class F>
ScopeExit<F> scope_exit(F f) { return ScopeExit<F>{f}; }

}  // namespace pipsort
