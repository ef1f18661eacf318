// Generic scoring path: ONE WARP per union configuration of up to KMAX SNPs.
//
// This is the device restatement of expand_and_compute_lkl (sss_postcal.cpp:447-685) and of the body
// of computeTotalLikelihood's loop (postcal.cpp:825-1044) for arbitrary union subsets.  It serves
//   * the stochastic shotgun search (one launch per neighbourhood, pipsort_score_union_configs),
//   * the exhaustive path for subset sizes the register kernel (exhaustive.cuh) does not cover,
//   * the parity tests as a second, independently written CUDA path.
//
// Per configuration (k union SNPs):
//   1. lanes gather the k x k causal sub-blocks of both studies' W = d Sigma~ into shared memory;
//   2. lane m computes E_s(mask m) for every sub-mask of the k SNPs (2^k Cholesky factorisations of
//      size <= k, in registers/local memory) -> shared-memory tables  (em, en, f) per study;
//   3. the 3^k expansions (mask pairs (m0,m1) with m0|m1 = all, postcal.cpp:903-958) are products of two
//      table entries; they are summed per (SNP, state) cell relative to the cell's structurally
//      largest term (see DESIGN.md "cells"), warp-reduced, and added to the bins;
//   4. the expansion with the largest |l| is returned (sss_postcal.cpp:624-626).
#pragma once
#include "common.cuh"

namespace pipsort {

typedef unsigned long long u64;

// ---- combinatorial unranking (replaces nextBinary / findConfig, postcal.cpp:307-387) ------------------
__device__ __forceinline__ u64 binom_dev(int n, int k) {
    if (k < 0 || k > n) return 0;
    unsigned __int128 v = 1;
    for (int i = 1; i <= k; i++) v = v * (unsigned)(n - k + i) / (unsigned)i;
    return (u64)v;
}

// r in [0, C(U,j)) -> the r-th j-subset of {0..U-1} in lexicographic order (ascending elements)
__device__ inline void unrank_subset(u64 r, int U, int j, int* g) {
    int x0 = 0;
    for (int i = 0; i < j; i++) {
        const int jj = j - i;
        const u64 base = binom_dev(U - x0, jj);
        int lo = x0, hi = U - jj;
        while (lo < hi) {  // largest x with #subsets whose i-th element is in [x0, x)  <=  r
            int mid = (lo + hi + 1) >> 1;
            if (base - binom_dev(U - mid, jj) <= r) lo = mid; else hi = mid - 1;
        }
        r -= base - binom_dev(U - lo, jj);
        g[i] = lo;
        x0 = lo + 1;
    }
}

// lexicographic successor; returns false after the last subset
__device__ inline bool next_subset(int U, int j, int* g) {
    int i = j - 1;
    while (i >= 0 && g[i] == U - j + i) i--;
    if (i < 0) return false;
    g[i]++;
    for (int t = i + 1; t < j; t++) g[t] = g[t - 1] + 1;
    return true;
}

// ---- per-warp shared-memory workspace -----------------------------------------------------------------
struct WarpWS {
    int* g;          // [KMAX] internal union indices
    int* loc;        // [2][KMAX]
    double* Wsub;    // [2][KMAX*KMAX]
    double* zs;      // [2][KMAX]
    double* em;      // [2][1<<kmax]
    double* f;       // [2][1<<kmax]
    int* en;         // [2][1<<kmax]
    int tabn;        // 1 << kmax
};

__host__ __device__ inline size_t warp_ws_bytes(int kmax) {
    size_t tabn = (size_t)1 << kmax;
    return 2 * KMAX * KMAX * 8 + 2 * KMAX * 8 + 2 * tabn * 8 * 2 + 2 * tabn * 4 + 3 * KMAX * 4 + 8;
}

__device__ inline WarpWS warp_ws(unsigned char* base, int kmax) {
    WarpWS w;
    w.tabn = 1 << kmax;
    double* d = reinterpret_cast<double*>(base);
    w.Wsub = d; d += 2 * KMAX * KMAX;
    w.zs = d; d += 2 * KMAX;
    w.em = d; d += 2 * w.tabn;
    w.f = d; d += 2 * w.tabn;
    int* i = reinterpret_cast<int*>(d);
    w.en = i; i += 2 * w.tabn;
    w.g = i; i += KMAX;
    w.loc = i;
    return w;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ int pow3(int k) {
    int v = 1;
    for (int i = 0; i < k; i++) v *= 3;
    return v;
}

// Scores the configuration whose internal union indices are in ws.g[0..k).  Warp-collective.
// Returns (on every lane) the expansion value l with the largest |l|, 0.0 if there is none.
// SK != STORE_PLAIN: class-resolved store (PIPSORT_PRIOR_CLASSES, common.cuh): the cells are kept per a' = a - [t == 2]
// instead of being weighted with L.pi[k][a], and go unweighted to their (k, t, a') slots; the total per a, the no-causal sums
// per class.  STORE_COUNTS: the total also per (a, b0), b0 = popcount(m0) - a, into the count table.
template <StoreKind SK = STORE_PLAIN>
__device__ inline double score_config(const LocusDev& L, const WarpWS& ws, int k, bool upd, int lane) {
    constexpr bool CR = SK != STORE_PLAIN;
    const AccDev& acc = L.acc;
    if (k == 0) {  // postcal.cpp:793-822, sss_postcal.cpp:463-499
        if (upd && lane == 0) {
            const double einv = 0.36787944117144233;  // exp(-1): the "- sqrt(|1|)" of postcal.cpp:802
            if (CR) {
                scal_add(acc, cls_T(0, 0), einv, 0);
                scal_add(acc, cls_N(acc.ccls, 0, 0), einv, 0);
                scal_add(acc, cls_N(acc.ccls, 1, 0), einv, 0);
                if (SK == STORE_COUNTS) scal_add(acc, cls_R(acc.ccls, 0, 0, 0), einv, 0);
            } else {
                bin_add(acc, SCAL, S_TOTAL, einv, 0);
                bin_add(acc, SCAL, S_NC0, einv, 0);
                bin_add(acc, SCAL, S_NC1, einv, 0);
            }
            count_add(acc, 1ull);
        }
        return L.null_l;
    }
    const int FULL = (1 << k) - 1;
    // 1. study-local indices, presence masks, causal sub-blocks
    if (lane < 2 * k) {
        int s = lane / k, i = lane - s * k;
        ws.loc[s * KMAX + i] = L.loc[s][ws.g[i]];
    }
    __syncwarp();
    int P[2];
#pragma unroll
    for (int s = 0; s < 2; s++) {
        int here = (lane < k) && (ws.loc[s * KMAX + lane] >= 0);
        P[s] = (int)__ballot_sync(0xffffffffu, here);
    }
    for (int t = lane; t < 2 * k * k; t += 32) {
        int s = t / (k * k), r = t - s * k * k, a = r / k, b = r - a * k;
        int la = ws.loc[s * KMAX + a], lb = ws.loc[s * KMAX + b];
        double v = 0.0;
        if (la >= 0 && lb >= 0) v = L.st[s].W[(size_t)la * L.st[s].ldw + lb];
        ws.Wsub[s * KMAX * KMAX + a * KMAX + b] = v;
    }
    if (lane < 2 * k) {
        int s = lane / k, i = lane - s * k;
        int li = ws.loc[s * KMAX + i];
        ws.zs[s * KMAX + i] = li >= 0 ? L.st[s].z[li] : 0.0;
    }
    __syncwarp();
    // 2. E_s(mask) tables
    bool notpd = false;
    for (int t = lane; t < 2 * (FULL + 1); t += 32) {
        const int s = t / (FULL + 1), m = t - s * (FULL + 1);
        double em = 0.0, fv = 0.0;
        int en = 0;
        if ((m & ~P[s]) == 0) {
            if (m == 0) {
                em = 1.0;
            } else {
                const double* Ws = ws.Wsub + s * KMAX * KMAX;
                const double* zz = ws.zs + s * KMAX;
                int id[KMAX];
                int cnt = 0;
                for (int i = 0; i < k; i++) if (m >> i & 1) id[cnt++] = i;
                double Lp[KMAX * (KMAX + 1) / 2], y[KMAX];
                double q = 0.0, prodL = 1.0;
                for (int a = 0; a < cnt; a++) {
                    const int ra = a * (a + 1) / 2;
                    for (int b = 0; b <= a; b++) {
                        const int rb = b * (b + 1) / 2;
                        double sacc = Ws[id[a] * KMAX + id[b]] + (a == b ? 1.0 : 0.0);
                        for (int c = 0; c < b; c++) sacc -= Lp[ra + c] * Lp[rb + c];
                        if (a == b) {
                            if (!(sacc > 0.0)) { notpd = true; sacc = 1.0; }
                            double l = sqrt(sacc);
                            Lp[ra + a] = l;
                            prodL *= l;
                        } else {
                            Lp[ra + b] = sacc / Lp[rb + b];
                        }
                    }
                    double ya = zz[id[a]];
                    for (int c = 0; c < a; c++) ya -= Lp[ra + c] * y[c];
                    ya /= Lp[ra + a];
                    y[a] = ya;
                    q += ya * ya;
                }
                const double hq = L.st[s].hd * q;
                fv = hq - log(prodL);
                xexp(hq, em, en);
                em /= prodL;
            }
        }
        ws.em[s * ws.tabn + m] = em;
        ws.f[s * ws.tabn + m] = fv;
        ws.en[s * ws.tabn + m] = en;
    }
    if (__any_sync(0xffffffffu, notpd) && lane == 0) flag_set(acc, ERR_NOT_PD);
    __syncwarp();
    // exponent of an absent mask aliases the mask restricted to the SNPs the study has (mantissa stays 0)
    for (int t = lane; t < 2 * (FULL + 1); t += 32) {
        const int s = t / (FULL + 1), m = t - s * (FULL + 1);
        if (m & ~P[s]) ws.en[s * ws.tabn + m] = ws.en[s * ws.tabn + (m & P[s])];
    }
    __syncwarp();
    const double* em0 = ws.em;
    const double* em1 = ws.em + ws.tabn;
    const int* en0 = ws.en;
    const int* en1 = ws.en + ws.tabn;
    const uint32_t* tab = L.exptab[k];
    const int n3 = pow3(k);
    // 4. expansion with the largest |l|  (sss_postcal.cpp:560,624-626), and the number of expansions
    double best = 0.0;
    int beste = 0x7fffffff, nvalid = 0;
    for (int e = lane; e < n3; e += 32) {
        const uint32_t pk = tab[e];
        const int m0 = pk & 255, m1 = (pk >> 8) & 255, a = pk >> 16;
        if ((m0 & ~P[0]) || (m1 & ~P[1])) continue;
        nvalid++;
        const double l = (L.neg_half_K + (ws.f[m0] + ws.f[ws.tabn + m1])) + L.logprior[k][a];
        if (fabs(l) > fabs(best)) { best = l; beste = e; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ob = __shfl_xor_sync(0xffffffffu, best, o);
        int oe = __shfl_xor_sync(0xffffffffu, beste, o);
        if (fabs(ob) > fabs(best) || (fabs(ob) == fabs(best) && oe < beste)) { best = ob; beste = oe; }
        nvalid += __shfl_xor_sync(0xffffffffu, nvalid, o);
    }
    if (!upd || nvalid == 0) return best;
    // 3. cells
    const int n3m = n3 / 3;
    for (int i = 0; i < k; i++) {
        const int bit = 1 << i, g = ws.g[i], p3i = pow3(i);
        for (int t = 0; t < 3; t++) {  // 0: study 0 only, 1: study 1 only, 2: both  (digit order of postcal.cpp:930-943)
            const bool in0 = t != 1, in1 = t != 0;
            if ((in0 && !(P[0] & bit)) || (in1 && !(P[1] & bit))) continue;
            const int r0 = (in0 ? FULL : FULL ^ bit) & P[0], r1 = (in1 ? FULL : FULL ^ bit) & P[1];
            const int nr = en0[r0] + en1[r1];
            if constexpr (CR) {
                double sa[KMAX];                      // sa[a'] (registers: the index is resolved by the unrolled selects)
#pragma unroll
                for (int q = 0; q < KMAX; q++) sa[q] = 0.0;
                for (int ep = lane; ep < n3m; ep += 32) {
                    const int hi = ep / p3i, lo = ep - hi * p3i;
                    const uint32_t pk = tab[(hi * 3 + t) * p3i + lo];
                    const int m0 = pk & 255, m1 = (pk >> 8) & 255, ap = (int)(pk >> 16) - (t == 2 ? 1 : 0);
                    const double v0 = em0[m0], v1 = em1[m1];
                    if (v0 == 0.0 || v1 == 0.0) continue;
                    int de = en0[m0] + en1[m1] - nr;
                    de = min(de, 1000);
                    const double v = v0 * v1 * pow2c(max(de, -2000));
#pragma unroll
                    for (int q = 0; q < KMAX; q++) sa[q] += q == ap ? v : 0.0;
                }
#pragma unroll
                for (int q = 0; q < KMAX; q++) {
                    if (q >= k) break;
                    const double v = warp_sum(sa[q]);
                    if (lane == 0) {
                        bin_add(acc, cls_slot(k, t, q), g, v, nr);
                        if (i == 0) scal_add(acc, cls_T(k, q + (t == 2 ? 1 : 0)), v, nr);
                    }
                }
                if (SK == STORE_COUNTS && i == 0) {   // the same expansions by class (a, b0)
                    // sr[a (2k + 3 - a) / 2 + b0]: the classes of size k, each with its own exponent (a class may lie far below
                    // the cell's reference nr, where a plain sum relative to it would flush its terms)
                    XAcc sr[cls_ntab(KMAX)];
                    const int nl = cls_ntab(k);
                    for (int q = 0; q < nl; q++) sr[q] = xacc_empty();
                    for (int ep = lane; ep < n3m; ep += 32) {
                        const int hi = ep / p3i, lo = ep - hi * p3i;
                        const uint32_t pk = tab[(hi * 3 + t) * p3i + lo];
                        const int m0 = pk & 255, m1 = (pk >> 8) & 255, a = pk >> 16;
                        const double v0 = em0[m0], v1 = em1[m1];
                        if (v0 == 0.0 || v1 == 0.0) continue;
                        xadd(sr[a * (2 * k + 3 - a) / 2 + __popc(m0) - a], v0 * v1, en0[m0] + en1[m1]);
                    }
                    for (int q = 0; q < nl; q++) {
                        const XAcc v = xwarp_sum(sr[q]);
                        if (lane == 0) scal_add(acc, cls_R(acc.ccls, k, 0, 0) + q, v.M, v.N);
                    }
                }
                continue;
            }
            double sx = 0.0, sy = 0.0;
            for (int ep = lane; ep < n3m; ep += 32) {
                const int hi = ep / p3i, lo = ep - hi * p3i;
                const uint32_t pk = tab[(hi * 3 + t) * p3i + lo];
                const int m0 = pk & 255, m1 = (pk >> 8) & 255, a = pk >> 16;
                const double v0 = em0[m0], v1 = em1[m1];
                if (v0 == 0.0 || v1 == 0.0) continue;
                int de = en0[m0] + en1[m1] - nr;
                de = min(de, 1000);
                const double v = v0 * v1 * pow2c(max(de, -2000));
                sy += v;
                sx = fma(v, L.pi[k][a], sx);
            }
            sx = warp_sum(sx);
            sy = warp_sum(sy);
            if (lane == 0) {
                bin_add(acc, t == 0 ? X1 : (t == 1 ? X2 : X3), g, sx, nr);
                bin_add(acc, t == 2 ? YS : YN, g, sy, nr);
                if (i == 0) bin_add(acc, SCAL, S_TOTAL, sx, nr);
            }
        }
    }
    if (lane == 0) {  // no causal SNP in a study: the other study carries all k (postcal.cpp:988-1000)
        if (CR) {
            if ((FULL & ~P[0]) == 0) scal_add(acc, cls_N(acc.ccls, 1, k), em0[FULL], en0[FULL]);
            if ((FULL & ~P[1]) == 0) scal_add(acc, cls_N(acc.ccls, 0, k), em1[FULL], en1[FULL]);
        } else {
            if ((FULL & ~P[0]) == 0) bin_add(acc, SCAL, S_NC1, L.pi[k][0] * em0[FULL], en0[FULL]);
            if ((FULL & ~P[1]) == 0) bin_add(acc, SCAL, S_NC0, L.pi[k][0] * em1[FULL], en1[FULL]);
        }
        count_add(acc, (u64)nvalid);
    }
    return best;
}

constexpr int SCORE_WARPS = 8;

// Batch of union configurations in snp_map (user) order, -1 padded.
__global__ void __launch_bounds__(SCORE_WARPS * 32)
score_batch_kernel(LocusDev L, const int* __restrict__ idx, long long n, int kmax, int ws_kmax,
                   const unsigned char* __restrict__ make_updates, double* __restrict__ out, const int* __restrict__ n_extra) {
    extern __shared__ __align__(16) unsigned char smem[];
    if (n_extra) n += *n_extra;          // batch length decided on the device (sss.cuh: 1 + number of unseen neighbours)
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    WarpWS ws = warp_ws(smem + (size_t)wib * warp_ws_bytes(ws_kmax), ws_kmax);
    const long long nw = (long long)gridDim.x * SCORE_WARPS;
    for (long long c = (long long)blockIdx.x * SCORE_WARPS + wib; c < n; c += nw) {
        int v = -1;
        if (lane < kmax) v = idx[c * kmax + lane];
        const unsigned present = __ballot_sync(0xffffffffu, v >= 0);
        const int k = __popc(present);
        // a row must list distinct union SNPs in increasing order, all below U (the reference builds its rows that way,
        // sss_postcal.cpp:20-99); anything else is refused like a bad explicit configuration (given.cuh)
        int prev = -1;
        {
            const unsigned below = present & ((1u << lane) - 1);
            const int src = below ? 31 - __clz(below) : lane;
            const int pv = __shfl_sync(0xffffffffu, v, src);
            if (below) prev = pv;
        }
        const bool bad_row = __any_sync(0xffffffffu, v >= 0 && (v >= L.U || v <= prev));
        if (bad_row) {
            if (lane == 0) { flag_set(L.acc, ERR_BAD_CONFIG); if (out) out[c] = 0.0; }
            continue;
        }
        if (v >= 0) ws.g[__popc(present & ((1u << lane) - 1))] = L.u2i[v];
        __syncwarp();
        const bool upd = make_updates ? make_updates[c] != 0 : true;
        const double best = score_config(L, ws, k, upd, lane);
        if (lane == 0 && out) out[c] = best;
        __syncwarp();
    }
}

// Exhaustive enumeration of the j-subsets with in-class ranks [r_begin, r_end) (internal SNP order):
// every warp takes chunks of `chunk` consecutive ranks, unranks the first and walks the rest.
// SK: the engine's store (StoreKind, common.cuh); the engine launches the instantiation that matches it.
template <StoreKind SK>
__global__ void __launch_bounds__(SCORE_WARPS * 32)
exhaustive_generic_kernel(LocusDev L, int j, u64 r_begin, u64 r_end, int chunk, int ws_kmax) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    WarpWS ws = warp_ws(smem + (size_t)wib * warp_ws_bytes(ws_kmax), ws_kmax);
    const u64 nchunks = (r_end - r_begin + chunk - 1) / chunk;
    const u64 nw = (u64)gridDim.x * SCORE_WARPS;
    for (u64 c = (u64)blockIdx.x * SCORE_WARPS + wib; c < nchunks; c += nw) {
        const u64 lo = r_begin + c * chunk;
        const u64 hi = min(lo + (u64)chunk, r_end);
        if (lane == 0) unrank_subset(lo, L.U, j, ws.g);
        __syncwarp();
        for (u64 r = lo; r < hi; r++) {
            score_config<SK>(L, ws, j, true, lane);
            __syncwarp();
            if (lane == 0) next_subset(L.U, j, ws.g);
            __syncwarp();
        }
    }
}

// Debug / parity: configuration at (rank, expansion) in the REFERENCE order over the snp_map order.
__global__ void enumerate_kernel(int U, const int* __restrict__ snp_map, int c, u64 rank, unsigned expansion,
                                 int* __restrict__ out_idx, int* __restrict__ out_state, unsigned* __restrict__ out_nexp) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int j = 0;
    for (; j <= c; j++) {  // size class, postcal.cpp:723-725
        u64 cnt = binom_dev(U, j);
        if (rank < cnt) break;
        rank -= cnt;
    }
    int g[KMAX];
    for (int i = 0; i < c; i++) { out_idx[i] = -1; out_state[i] = 0; }
    if (j > c) { *out_nexp = 0; return; }
    unrank_subset(rank, U, j, g);
    unsigned nexp = j == 0 ? 1u : 1u;
    bool ok = true;
    for (int i = 0; i < j; i++) {
        const bool h0 = snp_map[g[i]] >= 0, h1 = snp_map[U + g[i]] >= 0;
        if (h0 && h1) nexp *= 3u;
        if (!h0 && !h1) ok = false;
    }
    if (!ok) nexp = 0;
    *out_nexp = nexp;
    unsigned e = expansion;
    for (int i = 0; i < j; i++) {  // lowest chosen union SNP is the fastest digit (SURVEY.md H3)
        out_idx[i] = g[i];
        const bool h0 = snp_map[g[i]] >= 0, h1 = snp_map[U + g[i]] >= 0;
        int st = 0;
        if (h0 && h1) { st = 1 + (int)(e % 3u); e /= 3u; }
        else if (h0) st = 1;
        else if (h1) st = 2;
        out_state[i] = expansion < nexp ? st : 0;
    }
}

}  // namespace pipsort
