// Scoring path for batches of union configurations of up to LANE_KMAX SNPs: a PAIR OF LANES per configuration.
//
// Device restatement of a batch of expand_and_compute_lkl calls (sss_postcal.cpp:447-685, the body of the OpenMP loop
// sss_postcal.cpp:223-255): the stochastic shotgun search scores every neighbourhood with one launch of this kernel.
// The warp-per-configuration kernel of score.cuh left half of its lanes idle for k <= 4, factorised every one of the
// 2^k causal sub-blocks from scratch and walked all 3^k expansions per (SNP, state) cell.  Here, per configuration:
//
//   1. gather   the k(k-1)/2 + 2k entries of W = d Sigma~, A, z of a study -- the even lane of the pair takes study 0, the
//               odd lane study 1 (neighbours of one search state share all but one SNP, so the rows are L1/L2 hits: HBM
//               sees the LD rows of the current state once per launch);
//   2. tables   E_s(mask) for all 2^k sub-masks by BORDERING along a depth-first walk of the subset lattice: every mask
//               costs one row of forward substitution against its parent's Cholesky factor + one rsqrt + one exp
//               (fully unrolled per k: the factor lives in registers); the tables go to shared memory [study][mask][slot];
//   3. cells    the sum over the 3^k expansions (mask pairs with m0 | m1 = all, postcal.cpp:903-958) factorises because
//               the prior does: pi'(k, a) = pi'(k, 0) rho^a with a = |m0| + |m1| - k, rho = p / ((1 - p)/2).  With
//               g[m1] = rho^|m1| E_1[m1] and its superset sums Z[c] = sum_{m1 >= c} g[m1] (a zeta transform, k 2^(k-1)
//               additions) the total is sum_m0 rho^|m0| E_0[m0] Z[~m0] -- 2^k terms instead of 3^k -- and the per-SNP
//               cells (study 0 only / study 1 only / both) are the same sums with the transform left out along that
//               SNP's axis.  Only additions of non-negative terms: no cancellation.  The 2k (weighting, SNP) tasks of a
//               configuration are dealt to its two lanes; weighting and SNP are data, so the lanes run the same code;
//   4. max |l|  (sss_postcal.cpp:624-626) is attained at the largest or the smallest expansion weight: superset max / min
//               transforms of the same tables (one lane each), one log each;
//   5. update   the cells of one SNP are summed over the warp (a neighbourhood adds ~10^5 terms to the cells of the
//               4-5 SNPs of the current state) and leave it as one set of native fp64 atomics per SNP and warp.
//
// Numeric range: everything above is ordinary doubles, valid while every E_s(mask) < 2^450 (DESIGN.md "range").  A
// configuration that meets a larger value is handed to the mantissa/exponent code of score.cuh (whole warp, rare).
// Loci with p == 1 (rho infinite), priors under which the weights below leave the double range (engine.cu lane_peak_bits)
// and batches with more than LANE_KMAX SNPs per configuration use score.cuh throughout.
#pragma once
#include "exhaustive_dev.cuh"
#include "score.cuh"

namespace pipsort {

constexpr int LANE_KMAX = 5;
constexpr int LANE_WARPS = 4;
constexpr int LANE_THREADS = LANE_WARPS * 32;
constexpr int LANE_TAB = 1 << LANE_KMAX;        // masks per table
#ifndef LANE_DIAG
#define LANE_DIAG 0          // measurement builds only: 1 = no atomics leave the warp, 2 = tables only (no cells either)
#endif
#ifndef LANE_MINBLOCKS
#define LANE_MINBLOCKS 3
#endif

struct LaneBlockShared {
    double scal[3];                             // total, noCausal[0], noCausal[1] of the block (one lane per warp adds)
    double cnt;
};
constexpr int LANE_SLOTS = 16;                  // configurations per warp-step (two lanes each)
constexpr int LANE_CFG_PER_BLOCK = LANE_WARPS * LANE_SLOTS;
constexpr size_t LANE_TAB_BYTES = (size_t)LANE_WARPS * 2 * LANE_TAB * LANE_SLOTS * sizeof(double);    // [warp][study][mask][slot]
constexpr size_t LANE_CELL_BYTES = (size_t)LANE_WARPS * LANE_KMAX * 5 * LANE_SLOTS * sizeof(double);  // [warp][position][cell][slot]
constexpr size_t LANE_SMEM_BYTES = LANE_TAB_BYTES + LANE_CELL_BYTES + sizeof(LaneBlockShared);

template <int K>
struct LaneStudy {                              // causal sub-block of one study, positions 0..K-1 (virtual: W = 0, A = 1, z = 0)
    double w[K > 1 ? K * (K - 1) / 2 : 1];      // W[i][j], i < j, at j (j - 1) / 2 + i
    double A[K], z[K];
};

__host__ __device__ constexpr int lane_tri(int i, int j) { return j * (j - 1) / 2 + i; }
__host__ __device__ constexpr int lane_nth_bit(int mask, int j) {
    for (int b = 0; b < 31; b++)
        if (mask >> b & 1) { if (j == 0) return b; j--; }
    return 0;
}

template <int K>
struct LaneDfsCtx {
    const LaneStudy<K>& S;
    double hd;
    double* tab;            // &table[study][0][slot]; stride LANE_SLOTS doubles per mask
    int absent;             // positions the study does not have: masks touching them hold 0
    double Lr[K][K];        // chain rows: Lr[d][j], j < d
    double inv[K], y[K];
    double emax;
    int bad;
};

// children MASK | 1 << h, h = H .. K-1, of the node MASK (D = popcount(MASK) elements on the chain, all below H)
template <int K, int MASK, int D, int H>
struct LaneVisit {
    static __device__ __forceinline__ void run(LaneDfsCtx<K>& c, const double Eparent) {
        if constexpr (H < K) {
            constexpr int CH = MASK | (1 << H);
            double s = c.S.A[H], r = c.S.z[H];
            double v[D > 0 ? D : 1];
#pragma unroll
            for (int j = 0; j < D; j++) {
                double t = c.S.w[lane_tri(lane_nth_bit(MASK, j), H)];
#pragma unroll
                for (int i = 0; i < j; i++) t = fma(-v[i], c.Lr[j][i], t);
                t *= c.inv[j];
                v[j] = t;
                s = fma(-t, t, s);
                r = fma(-t, c.y[j], r);
            }
            c.bad |= !(s > 0.25);                 // A >= I: every Schur complement is >= 1 (postcal.cpp:291-294)
            const double rs = rsqrt_fast(s);
            const double u = r * rs;
            const double E = Eparent * (exp_pos(c.hd * (u * u)) * rs);
            c.emax = fmax(c.emax, E);
            c.tab[CH * LANE_SLOTS] = (CH & c.absent) ? 0.0 : E;
            if constexpr (H + 1 < K) {            // descend: the new element becomes chain row D
#pragma unroll
                for (int j = 0; j < D; j++) c.Lr[D][j] = v[j];
                c.inv[D] = rs;
                c.y[D] = u;
                LaneVisit<K, CH, D + 1, H + 1>::run(c, E);
            }
            LaneVisit<K, MASK, D, H + 1>::run(c, Eparent);
        }
    }
};

// superset sums / max / min along every axis of a 2^K array except axis SKIP (SKIP = -1: all axes)
template <int K, int SKIP, class Op>
__device__ __forceinline__ void lane_zeta(double (&z)[1 << K], Op op) {
#pragma unroll
    for (int a = 0; a < K; a++) {
        if (a == SKIP) continue;
#pragma unroll
        for (int c = 0; c < (1 << K); c++)
            if (!(c >> a & 1)) z[c] = op(z[c], z[c | (1 << a)]);
    }
}

// Cells of SNP i from the two tables of a configuration: {study 0 only, study 1 only, both}.  i is a RUN-TIME value (the
// loop over the SNPs is not unrolled: straight-line code for every SNP of every k made the kernel instruction-fetch
// bound); the tables are read through the bit permutation that moves SNP i to the top bit, where the code is the same for
// all i.  sc0 / sc1: weights per popcount of the mask (all ones for the likelihood-only sums).
template <int K>
__device__ __forceinline__ void lane_cells_one(const double* __restrict__ t0, const double* __restrict__ t1, const int i,
                                               const double (&sc0)[K + 1], const double (&sc1)[K + 1],
                                               double& x1, double& x2, double& x3) {
    constexpr int NM = 1 << K, H = NM >> 1;
    const int low = (1 << i) - 1, bi = 1 << i;
    double z[NM];
#pragma unroll
    for (int c = 0; c < H; c++) {
        const int m = (c & low) | ((c & ~low) << 1);        // mask of the other SNPs, SNP i left out
        const int pc = __popc(c);                           // compile-time after unrolling; the permutation keeps it
        z[c] = t1[m * LANE_SLOTS] * sc1[pc];
        z[c | H] = t1[(m | bi) * LANE_SLOTS] * sc1[pc + 1];
    }
    lane_zeta<K, K - 1>(z, [](double a, double q) { return a + q; });   // z[c] = sum over m1 >= c that agree with c on SNP i
    x1 = 0.0; x2 = 0.0; x3 = 0.0;
#pragma unroll
    for (int r0 = 0; r0 < H; r0++) {
        const int m = (r0 & low) | ((r0 & ~low) << 1);
        const int pc = __popc(r0);
        const double eo = t0[m * LANE_SLOTS] * sc0[pc], ew = t0[(m | bi) * LANE_SLOTS] * sc0[pc + 1];
        const int cmp = (H - 1) ^ r0;                       // the other SNPs that study 1 must carry
        x1 = fma(ew, z[cmp], x1);                           // i in study 0 only
        x2 = fma(eo, z[cmp | H], x2);                       // i in study 1 only
        x3 = fma(ew, z[cmp | H], x3);                       // i in both
    }
}

// Cells of the warp's configurations (shared-memory scratch cellw[(position * 5 + cell) * LANE_SLOTS + slot]) ->
// accumulator store.  The configurations of a neighbourhood share all but one SNP (sss_postcal.cpp:20-99), so ~10^5 terms
// of one launch go to the cells of the 4-5 SNPs of the current state.  The SNPs of the first two configurations (two
// neighbours drop different SNPs of the state, so together they name all of it) are tried as keys: a key held by at
// least four configurations is summed over the warp and leaves it as ONE set of native fp64 atomics; everything else
// goes out configuration by configuration, mostly to distinct addresses.  Warp-collective; pending = positions of this
// lane that still have to be flushed (0 on the odd lanes: the even lane of a pair flushes).
template <int K>
__device__ __forceinline__ void lane_flush_cells(const AccDev& acc, const int lane, const int (&g)[LANE_KMAX], int pending,
                                                 const double* __restrict__ cellw) {
    const int slot = lane >> 1;
#pragma unroll 1
    for (int it = 0; it < 2 * K; it++) {
        int mykey = -1;
#pragma unroll
        for (int i = 0; i < K; i++) if (i == (it >= K ? it - K : it)) mykey = (pending >> i & 1) ? g[i] : -1;
        const int key = __shfl_sync(0xffffffffu, mykey, it >= K ? 2 : 0);
        if (key < 0) continue;
        int pos = -1;
#pragma unroll
        for (int i = 0; i < K; i++) if ((pending >> i & 1) && g[i] == key) pos = i;
        const unsigned holders = __ballot_sync(0xffffffffu, pos >= 0);
        if (__popc(holders) < 4) continue;
        double mine = 0.0;
#pragma unroll
        for (int q = 0; q < 5; q++) {
            double r = pos >= 0 ? cellw[(pos * 5 + q) * LANE_SLOTS + slot] : 0.0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
            if (lane == q) mine = r;
        }
        if (lane < 5) bin_add(acc, lane, key, mine, 0);
        if (pos >= 0) pending &= ~(1 << pos);
    }
#pragma unroll 1
    for (int i = 0; i < K; i++)
        if (pending >> i & 1) {
            int gi = 0;
#pragma unroll
            for (int q = 0; q < K; q++) if (q == i) gi = g[q];
#pragma unroll
            for (int q = 0; q < 5; q++) bin_add(acc, q, gi, cellw[(i * 5 + q) * LANE_SLOTS + slot], 0);
        }
}

// One warp-step: LANE_SLOTS configurations, all with at most K SNPs (K = the largest k of the warp; shorter ones are
// padded with virtual SNPs that exist in study 0 only and carry no weight).  g[i] = internal union index of position i
// (i < k); both lanes of a pair hold the same g, k, live, upd.
template <int K>
__device__ __forceinline__ void lane_score(const LocusDev& L, LaneBlockShared& B, double* __restrict__ tabw, double* __restrict__ cellw,
                                           const int lane, const int (&g)[LANE_KMAX], const int k, const bool live, const bool upd,
                                           double& best, bool& slow) {
    constexpr int NM = 1 << K, FULL = NM - 1;
    const AccDev& acc = L.acc;
    const int role = lane & 1, slot = lane >> 1;
    double* t0 = tabw + slot;
    double* t1 = tabw + LANE_TAB * LANE_SLOTS + slot;
    const int padmask = FULL & ~((1 << k) - 1);
    int pres0, pres1;
    double emax;
    int bad;
    {   // ---- this lane's study: gather + table -----------------------------------------------------------------------
        const StudyDev& S = L.st[role];
        LaneStudy<K> T;
        int loc[K];
        int ps = 0;
#pragma unroll
        for (int i = 0; i < K; i++) {
            loc[i] = i < k ? L.loc[role][g[i]] : -1;
            const bool h = loc[i] >= 0;
            ps |= h ? (1 << i) : 0;
            T.A[i] = h ? S.A[loc[i]] : 1.0;
            T.z[i] = h ? S.z[loc[i]] : 0.0;
        }
#pragma unroll
        for (int j = 1; j < K; j++)
#pragma unroll
            for (int i = 0; i < j; i++) {
                const bool h = loc[i] >= 0 && loc[j] >= 0;
                const int lo = min(loc[i], loc[j]), hi = max(loc[i], loc[j]);
                T.w[lane_tri(i, j)] = h ? S.W[(size_t)lo * S.ldw + hi] : 0.0;
            }
        LaneDfsCtx<K> c{T, S.hd, role == 0 ? t0 : t1, FULL & ~(ps | (role == 0 ? padmask : 0)), {}, {}, {}, 0.0, 0};
        c.tab[0] = 1.0;
        LaneVisit<K, 0, 0, 0>::run(c, 1.0);
        const int po = __shfl_xor_sync(0xffffffffu, ps, 1);
        pres0 = role == 0 ? ps : po;
        pres1 = role == 0 ? po : ps;
        emax = fmax(c.emax, __shfl_xor_sync(0xffffffffu, c.emax, 1));
        bad = c.bad | __shfl_xor_sync(0xffffffffu, c.bad, 1);
    }
    __syncwarp();                                 // both tables of every configuration are in shared memory
    slow = live && (bad || !(emax < FAST_LIMIT));
    best = 0.0;
    int nvalid = 1;
#pragma unroll
    for (int i = 0; i < K; i++)
        if (i < k) nvalid *= ((pres0 >> i & 1) && (pres1 >> i & 1)) ? 3 : (((pres0 | pres1) >> i & 1) ? 1 : 0);
    // a SNP that exists in neither study: no expansion passes checkOR -> nothing to score
    const bool go = live && !slow && nvalid > 0;
    const bool acc_on = go && upd;
    double tot = 0.0, nc0 = 0.0, nc1 = 0.0, lmine = 0.0;
    // prior weights per popcount: study 0 side pi'(k,0) rho^(|m0| - K), study 1 side rho^|m1|  (pads count in |m0| only)
    double w0[K + 1], w1[K + 1];
    {
        w1[0] = 1.0;
#pragma unroll
        for (int j = 1; j <= K; j++) w1[j] = w1[j - 1] * L.rho;
        const double cx = L.pi[k][0] / w1[K];
#pragma unroll
        for (int j = 0; j <= K; j++) w0[j] = cx * w1[j];
    }
    if (go) {
        {   // max |l| over the expansions: at the largest weight (even lane) or the smallest (odd lane: a maximum of negated
            // values, so that both lanes run one piece of code)
            const double ninf = __longlong_as_double(0xfff0000000000000ll);
            double z[NM];
#pragma unroll
            for (int m = 0; m < NM; m++) {
                const double v = t1[m * LANE_SLOTS] * w1[__popc(m)];
                z[m] = role ? (v > 0.0 ? -v : ninf) : v;
            }
            lane_zeta<K, -1>(z, [](double a, double q) { return fmax(a, q); });
            double vb = ninf;
#pragma unroll
            for (int m0 = 0; m0 < NM; m0++) {
                const double e = t0[m0 * LANE_SLOTS] * w0[__popc(m0)];
                const double pr = e * z[FULL ^ m0];
                vb = fmax(vb, (role && !(e > 0.0)) ? ninf : pr);     // (0 * -inf is NaN)
            }
            lmine = L.cx + log(role ? -vb : vb);
        }
        if (upd && LANE_DIAG < 2) {
            // 2k tasks (weighting, SNP): t < k prior-weighted cells of SNP t (postValues / sharedPips, postcal.cpp:1003-1030),
            // t >= k likelihood-only cells of SNP t - k (sharedLL / notSharedLL, :1003-1016); dealt alternately to the two lanes
#pragma unroll 1
            for (int t = role; t < 2 * k; t += 2) {
                const bool weighted = t < k;
                const int i = weighted ? t : t - k;
                double s0[K + 1], s1[K + 1];
#pragma unroll
                for (int j = 0; j <= K; j++) { s0[j] = weighted ? w0[j] : 1.0; s1[j] = weighted ? w1[j] : 1.0; }
                double x1, x2, x3;
                lane_cells_one<K>(t0, t1, i, s0, s1, x1, x2, x3);
                if (weighted) {
                    cellw[(i * 5 + X1) * LANE_SLOTS + slot] = x1;
                    cellw[(i * 5 + X2) * LANE_SLOTS + slot] = x2;
                    cellw[(i * 5 + X3) * LANE_SLOTS + slot] = x3;
                    if (i == 0) tot = (x1 + x2) + x3;   // every expansion has SNP 0 in exactly one state: the total
                } else {
                    cellw[(i * 5 + YS) * LANE_SLOTS + slot] = x3;
                    cellw[(i * 5 + YN) * LANE_SLOTS + slot] = x1 + x2;
                }
            }
            if (role == 0) {   // noCausal: the other study carries every SNP (postcal.cpp:988-1000)
                nc1 = (t0[FULL * LANE_SLOTS] * w0[K]) * t1[0];
                nc0 = (t0[padmask * LANE_SLOTS] * w0[K - k]) * (t1[(FULL ^ padmask) * LANE_SLOTS] * w1[k]);
            }
        }
    }
    __syncwarp();                                 // the cells of a configuration were written by both of its lanes
    {   // (warp-collective code stays outside the per-configuration branches)
        const double other = __shfl_xor_sync(0xffffffffu, lmine, 1);
        const double lhi = role ? other : lmine, llo = role ? lmine : other;
        if (go) best = fabs(lhi) > fabs(llo) ? lhi : llo;
    }
    // ---- out of the warp: cells per SNP, scalars per warp -----------------------------------------------------------
    if (LANE_DIAG == 0 && __any_sync(0xffffffffu, acc_on)) {
        lane_flush_cells<K>(acc, lane, g, (acc_on && role == 0) ? ((1 << k) - 1) : 0, cellw);
        double r[4] = {tot, nc0, nc1, (acc_on && role == 0) ? (double)nvalid : 0.0};
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int q = 0; q < 4; q++) r[q] += __shfl_xor_sync(0xffffffffu, r[q], o);
        if (lane == 0) {
            atomicAdd(&B.scal[S_TOTAL], r[0]); atomicAdd(&B.scal[S_NC0], r[1]); atomicAdd(&B.scal[S_NC1], r[2]);
            atomicAdd(&B.cnt, r[3]);
        }
    }
}

// Batch of union configurations in snp_map (user) order, -1 padded, kmax <= LANE_KMAX columns.
__global__ void __launch_bounds__(LANE_THREADS, LANE_MINBLOCKS)
score_lane_kernel(LocusDev L, const int* __restrict__ idx, long long n, int kmax, const unsigned char* __restrict__ make_updates,
                  double* __restrict__ out, const int* __restrict__ n_extra) {
    extern __shared__ __align__(16) unsigned char smem[];
    double* tabs = reinterpret_cast<double*>(smem);
    LaneBlockShared& B = *reinterpret_cast<LaneBlockShared*>(smem + LANE_TAB_BYTES + LANE_CELL_BYTES);
    if (n_extra) n += *n_extra;          // batch length decided on the device (sss.cuh: 1 + number of unseen neighbours)
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    double* tabw = tabs + (size_t)wib * 2 * LANE_TAB * LANE_SLOTS;
    double* cellw = reinterpret_cast<double*>(smem + LANE_TAB_BYTES) + (size_t)wib * LANE_KMAX * 5 * LANE_SLOTS;
    if (threadIdx.x < 3) B.scal[threadIdx.x] = 0.0;
    if (threadIdx.x == 3) B.cnt = 0.0;
    __syncthreads();
    const long long nchunk = (n + LANE_CFG_PER_BLOCK - 1) / LANE_CFG_PER_BLOCK;
    for (long long ch = blockIdx.x; ch < nchunk; ch += gridDim.x) {
        const long long c = ch * LANE_CFG_PER_BLOCK + wib * LANE_SLOTS + (lane >> 1);     // both lanes of a pair: the same row
        const bool writer = (lane & 1) == 0;
        bool live = c < n;
        int g[LANE_KMAX];
        int k = 0;
        bool badrow = false;
        if (live) {
            int prev = -1;
#pragma unroll
            for (int i = 0; i < LANE_KMAX; i++) {
                g[i] = 0;
                const int v = i < kmax ? idx[c * kmax + i] : -1;
                if (v >= 0) {
                    // a row lists distinct union SNPs in increasing order, all below U (sss_postcal.cpp:20-99 builds them so)
                    if (v >= L.U || v <= prev) badrow = true;
                    else {
#pragma unroll
                        for (int q = 0; q < LANE_KMAX; q++) if (q == k) g[q] = L.u2i[v];
                        k++;
                    }
                    prev = v;
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < LANE_KMAX; i++) g[i] = 0;
        }
        const bool upd = live && (make_updates ? make_updates[c] != 0 : true);
        if (badrow) { if (writer) { flag_set(L.acc, ERR_BAD_CONFIG); if (out) out[c] = 0.0; } live = false; k = 0; }
        if (live && k == 0) {                       // the null configuration (sss_postcal.cpp:463-499)
            if (writer) {
                if (upd) {
                    const double einv = 0.36787944117144233;
                    atomicAdd(&B.scal[S_TOTAL], einv); atomicAdd(&B.scal[S_NC0], einv); atomicAdd(&B.scal[S_NC1], einv);
                    atomicAdd(&B.cnt, 1.0);
                }
                if (out) out[c] = L.null_l;
            }
            live = false;
        }
        const int kw = __reduce_max_sync(0xffffffffu, live ? k : 0);
        double best = 0.0;
        bool slow = false;
        switch (kw) {
            case 0: break;
            case 1: lane_score<1>(L, B, tabw, cellw, lane, g, k, live, upd, best, slow); break;
            case 2: lane_score<2>(L, B, tabw, cellw, lane, g, k, live, upd, best, slow); break;
            case 3: lane_score<3>(L, B, tabw, cellw, lane, g, k, live, upd, best, slow); break;
            case 4: lane_score<4>(L, B, tabw, cellw, lane, g, k, live, upd, best, slow); break;
            default: lane_score<5>(L, B, tabw, cellw, lane, g, k, live, upd, best, slow); break;
        }
        if (live && !slow && out && writer) out[c] = best;
        // configurations outside the plain-double range: the whole warp scores them one by one with the mantissa/exponent
        // code of score.cuh (its workspace aliases this warp's tables, which are dead by now)
        unsigned todo = __ballot_sync(0xffffffffu, slow && writer);
        if (todo) {
            __syncwarp();
            WarpWS ws = warp_ws(reinterpret_cast<unsigned char*>(tabw), LANE_KMAX);
            while (todo) {
                const int src = __ffs(todo) - 1;
                todo &= todo - 1;
                const int ks = __shfl_sync(0xffffffffu, k, src);
                const int us = __shfl_sync(0xffffffffu, (int)upd, src);
#pragma unroll
                for (int i = 0; i < LANE_KMAX; i++) {
                    const int gi = __shfl_sync(0xffffffffu, g[i], src);
                    if (lane == 0 && i < ks) ws.g[i] = gi;
                }
                __syncwarp();
                const double b = score_config(L, ws, ks, us != 0, lane);
                if (lane == src && out) out[c] = b;
                __syncwarp();
            }
        }
        __syncwarp();
    }
    __syncthreads();
    // the block's scalars: plain doubles relative to exponent 0
    if (threadIdx.x < 3) bin_add(L.acc, SCAL, threadIdx.x, B.scal[threadIdx.x], 0);
    if (threadIdx.x == 3 && B.cnt > 0.0) atomicAdd(L.acc.counters, B.cnt);
}

}  // namespace pipsort
