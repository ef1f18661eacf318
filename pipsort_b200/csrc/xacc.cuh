// Extended-range FP64 arithmetic for the PIPSORT posterior engine (sm_100a).
//
// The reference accumulates everything in log space (postcal.h:102-112, addlogSpace): one exp and
// one log per update, under an OpenMP critical section.  The raw-log outputs (shared_ll /
// notshared_ll columns, postcal.h:326) span thousands of nats inside one locus (tests/example:
// -43204 ... -40675), so a single linear scale cannot represent them in a double.  Here every
// weight exp(l) is carried as  m * 2^n  (m: non-negative double, n: int32) and every accumulator
// ("XAcc") as  M * 2^N ;  an update is one integer subtract, one exponent-field construction and
// one DFMA -- no exp, no log, no branch except the rare re-basing when a term is 2^512 larger than
// the accumulator's base.  Logs are taken once per accumulator in the finalize kernel.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace pipsort {

constexpr int XNEG = -(1 << 28);  // exponent of an "empty" value; 3*XNEG still fits in int32

struct XAcc {
    double M;
    int N;
};

__host__ __device__ __forceinline__ XAcc xacc_empty() { return XAcc{0.0, XNEG}; }

// 2^e for e in [-1022, 1023], +0.0 below (flush), caller guarantees e <= 1023
__device__ __forceinline__ double pow2c(int e) {
    int hi = max(e + 1023, 0) << 20;
    return __hiloint2double(hi, 0);
}

// acc += m * 2^n
__device__ __forceinline__ void xadd(XAcc& a, double m, int n) {
    int e = n - a.N;
    if (e > 512) {  // re-base on the new (much larger) term; old content is scaled down (maybe to 0)
        a.M *= pow2c(max(-e, -2000));
        a.N = n;
        e = 0;
    }
    a.M = fma(m, pow2c(e), a.M);
}

__device__ __forceinline__ void xmerge(XAcc& a, const XAcc& b) { xadd(a, b.M, b.N); }

// exp(t) = m * 2^n with m in [0.70, 1.42];  |t| < 2^30 ln 2.  Cody-Waite reduction + degree-13
// Taylor polynomial on |r| <= ln2/2 (truncation 4e-18 relative).  Coefficients live in constant memory so
// that the DFMAs take them as c[bank][offset] operands (no per-use UMOV pairs).
__constant__ double XEXP_C[12] = {
    1.6059043836821613e-10,   // 1/13!
    2.08767569878681e-09,     // 1/12!
    2.505210838544172e-08,    // 1/11!
    2.755731922398589e-07,    // 1/10!
    2.7557319223985893e-06,   // 1/9!
    2.48015873015873e-05,     // 1/8!
    1.984126984126984e-04,    // 1/7!
    1.3888888888888889e-03,   // 1/6!
    8.333333333333333e-03,    // 1/5!
    4.1666666666666664e-02,   // 1/4!
    1.6666666666666666e-01,   // 1/3!
    0.5};
__device__ __forceinline__ void xexp(double t, double& m, int& n) {
    const double LOG2E = 1.4426950408889634;
    const double LN2_HI = 6.93147180369123816490e-01;  // low 21 bits zero: k*LN2_HI exact for |k| < 2^21..
    const double LN2_LO = 1.90821492927058770002e-10;
    const double MAGIC = 6755399441055744.0;  // 1.5 * 2^52: rint + int extraction in one add
    double tmp = fma(t, LOG2E, MAGIC);
    n = __double2loint(tmp);
    double kf = tmp - MAGIC;
    double r = fma(-kf, LN2_HI, t);
    r = fma(-kf, LN2_LO, r);
#ifdef XEXP_HORNER
    double p = XEXP_C[0];
#pragma unroll
    for (int i = 1; i < 12; i++) p = fma(p, r, XEXP_C[i]);
    p = fma(p, r, 1.0);
    m = fma(p, r, 1.0);
#else
    // Estrin evaluation of sum_{i<=13} r^i / i!  (dependency depth 5 instead of 14)
    const double r2 = r * r;
    const double a0 = 1.0 + r;                         // c0 + c1 r
    const double a1 = fma(XEXP_C[10], r, XEXP_C[11]);  // 1/2! + r/3!
    const double a2 = fma(XEXP_C[8], r, XEXP_C[9]);    // 1/4! + r/5!
    const double a3 = fma(XEXP_C[6], r, XEXP_C[7]);    // 1/6! + r/7!
    const double a4 = fma(XEXP_C[4], r, XEXP_C[5]);    // 1/8! + r/9!
    const double a5 = fma(XEXP_C[2], r, XEXP_C[3]);    // 1/10! + r/11!
    const double a6 = fma(XEXP_C[0], r, XEXP_C[1]);    // 1/12! + r/13!
    const double r4 = r2 * r2;
    const double b0 = fma(a1, r2, a0);
    const double b1 = fma(a3, r2, a2);
    const double b2 = fma(a5, r2, a4);
    const double r8 = r4 * r4;
    const double d0 = fma(b1, r4, b0);
    const double d1 = fma(a6, r4, b2);
    m = fma(d1, r8, d0);
#endif
}

// two independent xexp evaluations written stage by stage: the scheduler keeps the order it is given as the tie-breaker,
// and one evaluation after the other would leave every dependent operation waiting out its full latency
__device__ __forceinline__ void xexp_pair(const double (&t)[2], double (&m)[2], int (&n)[2]) {
    const double LOG2E = 1.4426950408889634, LN2_HI = 6.93147180369123816490e-01, LN2_LO = 1.90821492927058770002e-10;
    const double MAGIC = 6755399441055744.0;
    double tmp[2], kf[2], r[2], r2[2], a[2][7], r4[2], b[2][3], r8[2], d[2][2];
#pragma unroll
    for (int s = 0; s < 2; s++) tmp[s] = fma(t[s], LOG2E, MAGIC);
#pragma unroll
    for (int s = 0; s < 2; s++) { n[s] = __double2loint(tmp[s]); kf[s] = tmp[s] - MAGIC; }
#pragma unroll
    for (int s = 0; s < 2; s++) r[s] = fma(-kf[s], LN2_HI, t[s]);
#pragma unroll
    for (int s = 0; s < 2; s++) r[s] = fma(-kf[s], LN2_LO, r[s]);
#pragma unroll
    for (int s = 0; s < 2; s++) {
        r2[s] = r[s] * r[s];
        a[s][0] = 1.0 + r[s];
#pragma unroll
        for (int i = 1; i < 7; i++) a[s][i] = fma(XEXP_C[12 - 2 * i], r[s], XEXP_C[13 - 2 * i]);
    }
#pragma unroll
    for (int s = 0; s < 2; s++) {
        r4[s] = r2[s] * r2[s];
        b[s][0] = fma(a[s][1], r2[s], a[s][0]);
        b[s][1] = fma(a[s][3], r2[s], a[s][2]);
        b[s][2] = fma(a[s][5], r2[s], a[s][4]);
    }
#pragma unroll
    for (int s = 0; s < 2; s++) {
        r8[s] = r4[s] * r4[s];
        d[s][0] = fma(b[s][1], r4[s], b[s][0]);
        d[s][1] = fma(a[s][6], r4[s], b[s][2]);
    }
#pragma unroll
    for (int s = 0; s < 2; s++) m[s] = fma(d[s][1], r8[s], d[s][0]);
}

// natural log of an accumulator; caller handles M == 0 (empty)
__device__ __forceinline__ double xlog(const XAcc& a) { return log(a.M) + (double)a.N * 0.6931471805599453094; }

// log(M 2^N) + c ; 0.0 (the reference's "empty" sentinel, postcal.h:102-112) when nothing was added
__device__ inline double xlog_or_zero(const XAcc& a, double c) {
    if (!(a.M > 0.0)) return 0.0;
    const double LN2_HI = 6.93147180369123816490e-01, LN2_LO = 1.90821492927058770002e-10;
    const double n = (double)a.N;
    return (n * LN2_HI + (log(a.M) + n * LN2_LO)) + c;
}

// warp-wide sum of XAccs: common exponent = max N over the warp (one REDUX), mantissas re-scaled
// to it (terms more than 2^1022 below the warp maximum flush to zero: they are below one ulp of
// the sum), then a plain shuffle tree.  Result valid in every lane.
__device__ __forceinline__ XAcc xwarp_sum(const XAcc& a) {
    int nmax = __reduce_max_sync(0xffffffffu, a.N);
    double v = a.M * pow2c(max(a.N - nmax, -2000));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return XAcc{v, nmax};
}

}  // namespace pipsort
