// Exhaustive path: device code in exhaustive_dev.cuh, work decomposition in exh_plan.h, planning + launch below.
#pragma once
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <tuple>
#include <vector>

#include "exhaustive_dev.cuh"

namespace pipsort {

struct ExhScratch {           // owned by the engine, reused across launches; the engine allocates both buffers
    int4* d_chunks = nullptr;     // chunk descriptors of the plan on the device
    size_t cap_chunks = 0;
    unsigned* d_counter = nullptr;   // [0] work-queue head, [1] finished blocks (the kernel re-arms both)
    int occ = 0;                  // resident blocks per SM of exhaustive_all_kernel
    char* pin_stage = nullptr;    // pinned staging slice for the FIRST descriptor upload (later ones may overlap an in-flight copy)
    size_t pin_stage_cap = 0;
    std::shared_ptr<const std::vector<ExhChunkDesc>> host_plan;   // keeps a pageable upload source alive
    // the plan of the last launch (a pass is usually repeated with the same c and rank range); valid once it is uploaded
    bool plan_valid = false;
    int plan_c = 0;
    unsigned long long plan_rb = 0, plan_re = 0;
    ExhAll plan;
    int plan_blocks = 0;
};

inline u64 exh_binom(int n, int k) {
    if (k < 0 || k > n) return 0;
    unsigned __int128 v = 1;
    for (int i = 1; i <= k; i++) v = v * (unsigned)(n - k + i) / (unsigned)i;
    return (u64)v;
}

inline void exh_unrank(u64 r, int U, int j, int* g) {
    int x0 = 0;
    for (int i = 0; i < j; i++) {
        const int jj = j - i;
        const u64 base = exh_binom(U - x0, jj);
        int lo = x0, hi = U - jj;
        while (lo < hi) {
            int mid = (lo + hi + 1) >> 1;
            if (base - exh_binom(U - mid, jj) <= r) lo = mid; else hi = mid - 1;
        }
        r -= base - exh_binom(U - lo, jj);
        g[i] = lo;
        x0 = lo + 1;
    }
}

// Fills the rank-range part of P for size class j; returns false when the class does not intersect.
inline bool exh_class_params(ExhParams& P, int U, int j, u64 rb, u64 re) {
    memset(&P, 0, sizeof P);
    P.J = j;
    if (U < j || rb >= re) return false;
    const u64 total = exh_binom(U, j);
    P.r_begin = rb; P.r_end = re;
    P.partial = !(rb == 0 && re == total);
    int glo[3] = {0, 0, 0}, ghi[3] = {U, U, U};
    exh_unrank(rb, U, j, glo);
    if (re < total) exh_unrank(re, U, j, ghi);
    for (int i = 0; i < 3; i++) { P.lo[i] = glo[i]; P.hi[i] = ghi[i]; }
    if (j == 3) {
        P.a_lo = glo[0];
        P.a_hi = std::min(re < total ? ghi[0] : U - 3, U - 3);
    } else {
        P.a_lo = P.a_hi = -1;
    }
    return true;
}

// Cost model of a locus (exh_plan.h); PIPSORT_EXH_COSTS="chain,plain,pair,pair1" overrides the measured constants (experiments).
inline ExhCostModel exh_cost_model(int U, const int* types) {
    ExhCostModel M(U, types);
    if (const char* v = getenv("PIPSORT_EXH_COSTS")) {
        double c[4] = {M.c_chain, M.c_plain, M.c_pair, M.c_pair1};
        sscanf(v, "%lf,%lf,%lf,%lf", &c[0], &c[1], &c[2], &c[3]);
        M.c_chain = c[0]; M.c_plain = c[1]; M.c_pair = c[2]; M.c_pair1 = c[3];
        for (double x : c) M.hash = (M.hash ^ (uint64_t)(x * 4096.0)) * 1099511628211ull;
    }
    return M;
}

// The chunk list for (U, class ranges, number of resident warps): pure arithmetic on U, so it is shared by every engine
// of the process (a fine-mapping run creates one engine per locus, and loci of equal size are common).
struct ExhPlanKey {
    int U, c, slots;
    u64 rb, re;
    double forced;
    u64 types;          // hash of the SNP-type layout (ExhCostModel): the step costs depend on it
    bool operator<(const ExhPlanKey& o) const {
        return std::tie(U, c, slots, rb, re, forced, types) < std::tie(o.U, o.c, o.slots, o.rb, o.re, o.forced, o.types);
    }
};

inline std::shared_ptr<const std::vector<ExhChunkDesc>> exh_plan_chunks(const ExhPlanKey& key, bool have3, const ExhParams& p3,
                                                                       bool have2, int n1_tiles, int tile1_0, int do_null,
                                                                       const ExhCostModel* M) {
    static std::map<ExhPlanKey, std::shared_ptr<const std::vector<ExhChunkDesc>>> cache;
    static std::mutex mu;
    {
        std::lock_guard<std::mutex> g(mu);
        auto it = cache.find(key);
        if (it != cache.end()) return it->second;
    }
    const int U = key.U;
    ExhCost cs;
    if (const char* v = getenv("PIPSORT_EXH_SETUP")) sscanf(v, "%lf,%lf,%lf,%lf", &cs.seg, &cs.win, &cs.a, &cs.chunk);   // experiments
    auto plan = std::make_shared<std::vector<ExhChunkDesc>>();
    const double steps = (have3 ? exh_class_steps(*M, 3, p3.a_lo, p3.a_hi, true) : 0.0) + (have2 ? exh_class_steps(*M, 2, 0, 0, true) : 0.0);
    // Granularity (measured on B200, scripts/sweep_chunks.py, scripts/trace_chunks.py).  avg = modelled cost per resident
    // warp, set-up work included (a chunk costs ~3 generic steps before its first step: measured 5.5 us against 1.3 us).
    //   avg <= 64 : ONE chunk per resident warp, all of the same cost -- a static, even deal: the kernel time of a small locus
    //               (or of a 1/8 shard of one: 1-3 steps per warp) is the time of its longest chunk, and a second chunk per
    //               warp would pay the set-up again;
    //   beyond    : ~avg / 32 (at most 12) chunks per resident warp, balanced by the work queue.
    const double setup = cs.chunk + cs.win + cs.seg + cs.a;
    double target = key.forced;
    if (!(target > 0.0)) {
        double avg = 1.15 * steps / key.slots + setup;
        for (int pass = 0; pass < 2 && avg <= 64.0; pass++) {     // set-up costs depend on the cuts: one refinement
            plan->clear();
            double tot = 0.0;
            if (have3) tot += exh_plan_class(*M, 3, p3.a_lo, p3.a_hi, avg, cs, *plan);
            if (have2) tot += exh_plan_class(*M, 2, 0, 0, avg, cs, *plan);
            avg = std::max(1.01 * tot / key.slots, setup + 1.0);
        }
        if (avg <= 64.0) target = avg;
        else target = avg / std::min(12.0, std::floor(avg / 32.0));
    }
    const bool one_round = !(key.forced > 0.0) && target <= 64.0 * 1.02;
    for (int tries = 0; tries < 8; tries++) {
        plan->clear();
        if (have3) exh_plan_class(*M, 3, p3.a_lo, p3.a_hi, target, cs, *plan);
        if (have2) exh_plan_class(*M, 2, 0, 0, target, cs, *plan);
        // one chunk per resident warp means AT MOST one: a handful of left-over chunks would cost a second round
        const double avail = (double)key.slots - n1_tiles - do_null;
        if (!one_round || avail < 1.0 || (double)plan->size() <= avail) break;
        target = std::max(target * 1.005 * std::max(1.0, (double)plan->size() / avail), target + 0.25);
    }
    if (one_round && plan->size() > 16) {
        // One chunk per resident warp: what a warp-step costs also depends on what the other warps of its SM are doing (three
        // warps share an FP64 pipe), and consecutive chunks are of the same kind -- the SMs that got the chunks among the
        // triples of three shared SNPs finished last (24 us of stepping against 16 for the median warp).  Deal the chunks out
        // with a stride, so that every CTA and every SM holds a mix.
        static const bool keep = getenv("PIPSORT_EXH_NO_SHUFFLE") != nullptr;
        if (!keep) {
            const size_t n = plan->size();
            size_t stride = (size_t)(0.6180339887 * (double)n) | 1;
            auto gcd = [](size_t a, size_t b) { while (b) { const size_t t = a % b; a = b; b = t; } return a; };
            while (gcd(stride, n) != 1) stride += 2;
            std::vector<ExhChunkDesc> mixed(n);
            for (size_t i = 0; i < n; i++) mixed[i] = (*plan)[(i * stride) % n];
            plan->swap(mixed);
        }
    }
    for (int t = 0; t < n1_tiles; t++) plan->push_back(ExhChunkDesc{tile1_0 + t, 0, 0, 1u << 28});
    if (do_null) plan->push_back(ExhChunkDesc{0, 0, 0, 0u});
    std::lock_guard<std::mutex> g(mu);
    if (cache.size() > 256) cache.clear();
    cache[key] = plan;
    return plan;
}

// The plan of ONE kernel for the size classes 0..min(c,3) restricted to the global union-subset rank range
// [rank_begin, rank_end) (size-then-lexicographic order over the internal SNP order).  Returns a cudaError_t.  Unless the
// plan of the last launch is reused, sc->plan.n_total descriptors then have to fit sc->d_chunks before exhaustive_launch.
inline int exhaustive_plan(const LocusDev& L, int c, u64 rank_begin, u64 rank_end, int sm_count, ExhScratch* sc,
                           const ExhCostModel* M) {
    const int U = L.U;
    cudaError_t err;
    // the instantiation that matches the engine's store (class-resolved: PIPSORT_PRIOR_CLASSES)
    const bool cr = L.acc.ccls > 0;
    if (!sc->occ) {
        void (*kernel)(LocusDev, ExhAll, const LocusDev*) = cr ? exhaustive_all_kernel<true> : exhaustive_all_kernel<false>;
        const size_t smem = cr ? EXH_SMEM_BYTES_CR : EXH_SMEM_BYTES;
        // (the attribute is per device: set it for every engine, not once per process)
        if ((err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return (int)err;
        static int occ_cache[2] = {0, 0};    // a property of the kernel and the device generation: query once per process
        static std::mutex occ_mutex;
        std::lock_guard<std::mutex> g(occ_mutex);
        if (!occ_cache[cr] && (err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_cache[cr], kernel, EXH_WARPS * 32, smem)) != cudaSuccess) return (int)err;
        sc->occ = occ_cache[cr];
    }
    const double forced = [] { const char* v = getenv("PIPSORT_EXH_CHUNK"); return v ? atof(v) : 0.0; }();   // experiments / tests
    if (sc->plan_valid && !(forced > 0.0) && sc->plan_c == c && sc->plan_rb == rank_begin && sc->plan_re == rank_end) return 0;
    ExhAll A;
    memset(&A, 0, sizeof A);
    u64 off = 0;
    bool have3 = false, have2 = false;
    int n1_tiles = 0, tile1_0 = 0, do_null = 0;
    for (int j = 0; j <= std::min(std::min(c, 3), U); j++) {
        const u64 cnt = exh_binom(U, j);
        const u64 lo = std::max<u64>(rank_begin, off), hi = std::min<u64>(rank_end, off + cnt);
        if (lo < hi) {
            const u64 rb = lo - off, re = hi - off;
            if (j == 0) do_null = 1;
            else if (j == 1) { A.x1_lo = (int)rb; A.x1_hi = (int)re; tile1_0 = A.x1_lo >> 5; n1_tiles = ((A.x1_hi - 1) >> 5) - tile1_0 + 1; }
            else if (j == 2) have2 = exh_class_params(A.p2, U, 2, rb, re);
            else have3 = exh_class_params(A.p3, U, 3, rb, re);
        }
        off += cnt;
    }
    const int occ = std::max(1, sc->occ);
    const int slots = sm_count * occ * EXH_WARPS;
    const ExhPlanKey key{U, c, slots, rank_begin, rank_end, forced > 0.0 ? forced : 0.0, M ? M->hash : 0};
    auto plan = exh_plan_chunks(key, have3, A.p3, have2, n1_tiles, tile1_0, do_null, M);
    if (plan->size() >= 0xfff00000ull) return (int)cudaErrorInvalidValue;   // 32-bit work queue (never in practice)
    A.n_total = (unsigned)plan->size();
    static const bool debug = getenv("PIPSORT_EXH_DEBUG") != nullptr;
    if (debug) {
        double st = 0; unsigned mx = 0;
        for (const ExhChunkDesc& d : *plan) { const unsigned n = d.nsteps_kind & 0x0fffffff; st += n; mx = std::max(mx, n); }
        fprintf(stderr, "[exhaustive] U=%d c=%d slots=%d chunks=%u steps=%.0f longest=%u cost3=%.0f\n", U, c, slots, A.n_total, st, mx,
                have3 ? exh_class_steps(*M, 3, A.p3.a_lo, A.p3.a_hi, true) : 0.0);
    }
    sc->host_plan = plan;                    // the upload may still be reading it after exhaustive_launch returns
    sc->plan = A;
    sc->plan_blocks = (int)std::min<u64>(((u64)A.n_total + EXH_WARPS - 1) / EXH_WARPS, (u64)sm_count * occ);
    sc->plan_valid = false; sc->plan_c = c; sc->plan_rb = rank_begin; sc->plan_re = rank_end;
    return 0;
}

// Uploads a new plan to sc->d_chunks and launches it.  Returns a cudaError_t.  ev0 / ev1 (optional) are recorded
// immediately around the kernel launch: the host-side planning is NOT part of the kernel's device time.
inline int exhaustive_launch(const LocusDev& L, const LocusDev* Lg, cudaStream_t stream, unsigned long long* launches, ExhScratch* sc,
                             cudaEvent_t ev0 = nullptr, cudaEvent_t ev1 = nullptr) {
    static_assert(sizeof(ExhChunkDesc) == sizeof(int4), "descriptor layout");
    cudaError_t err;
    if (!sc->plan_valid && sc->plan.n_total) {
        const size_t bytes = sc->host_plan->size() * sizeof(ExhChunkDesc);
        const void* src = sc->host_plan->data();
        if (sc->pin_stage && bytes <= sc->pin_stage_cap) {
            memcpy(sc->pin_stage, src, bytes);
            src = sc->pin_stage;
            sc->pin_stage = nullptr;             // one use
        }
        if ((err = cudaMemcpyAsync(sc->d_chunks, src, bytes, cudaMemcpyHostToDevice, stream)) != cudaSuccess) return (int)err;
        sc->plan.chunks = sc->d_chunks;
        sc->plan.counter = sc->d_counter;
    }
    sc->plan_valid = true;
    if (sc->plan.n_total == 0) return 0;
    const bool cr = L.acc.ccls > 0;
    if (ev0 && (err = cudaEventRecord(ev0, stream)) != cudaSuccess) return (int)err;
    if (cr) exhaustive_all_kernel<true><<<sc->plan_blocks, EXH_WARPS * 32, EXH_SMEM_BYTES_CR, stream>>>(L, sc->plan, Lg);
    else exhaustive_all_kernel<false><<<sc->plan_blocks, EXH_WARPS * 32, EXH_SMEM_BYTES, stream>>>(L, sc->plan, Lg);
    if (ev1 && (err = cudaEventRecord(ev1, stream)) != cudaSuccess) return (int)err;
    (*launches)++;
    return (int)cudaGetLastError();
}

}  // namespace pipsort
