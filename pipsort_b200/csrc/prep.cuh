// Locus pre-processing on the GPU: what Model does once per study before PostCal exists (model.h:171-264):
//   1. makeSigmaPositiveSemiDefinite (util.cpp:195-226): add 0.01 to the diagonal until the LU determinant is
//      > 0 (a determinant that underflows to 0 counts as "not positive": for thousands of SNPs the running product of
//      the pivots underflows, so the loop really runs dozens of times -- each pass is one O(n^3) LU);
//   2. eigen_decomp (util.cpp:228-263): Sigma + a I = Q Omega Q^T, |Omega| (model.h:227);
//   3. B = |Omega|^(1/2) Q^T, S' = |Omega|^(-1/2) Q^T z (model.h:230-255).
// What the engine needs from it (SURVEY.md section 0): the effective LD  B^T B = Q |Omega| Q^T
//   = (Sigma + a I) + 2 sum_{Omega_i < 0} |Omega_i| q_i q_i^T      (a rank-m correction, m = #negative eigenvalues,
//     0 whenever the shifted matrix is positive definite),
// z itself (B^T S' = z), and  K_s = S'^T S' = sum_i (q_i . z)^2 / |Omega_i|.
//
// The two dense factorizations are cuSOLVER's (Dgetrf: same partial-pivoting LU as GSL's gsl_linalg_LU_decomp, so the
// pivot sequence -- and with it the under/overflow behaviour of the determinant product -- is the reference's up to
// rounding; Dsyevd for the symmetric eigenproblem).  cuSOLVER is loaded lazily with dlopen so that the engine library
// itself has no link-time dependency on it; everything else (shift, determinant product in GSL's order, K, the
// negative-eigenvalue correction) is a small kernel below.  At 5000 SNPs/study the reference spends minutes here on the
// CPU (plus an unused 10^4 x 10^4 inverse in the PostCal constructor, postcal.h:186-187, which is not replicated).
#pragma once
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <string>

#include <cusolverDn.h>

#include "common.cuh"

namespace pipsort {

struct CusolverApi {
    void* lib = nullptr;
    decltype(&cusolverDnCreate) Create = nullptr;
    decltype(&cusolverDnDestroy) Destroy = nullptr;
    decltype(&cusolverDnSetStream) SetStream = nullptr;
    decltype(&cusolverDnDgetrf_bufferSize) Dgetrf_bufferSize = nullptr;
    decltype(&cusolverDnDgetrf) Dgetrf = nullptr;
    decltype(&cusolverDnDsyevd_bufferSize) Dsyevd_bufferSize = nullptr;
    decltype(&cusolverDnDsyevd) Dsyevd = nullptr;
    decltype(&cusolverDnDpotrf_bufferSize) Dpotrf_bufferSize = nullptr;
    decltype(&cusolverDnDpotrf) Dpotrf = nullptr;
    decltype(&cusolverDnDpotrs) Dpotrs = nullptr;
    bool ok = false, chol = false;
};

inline const CusolverApi& cusolver_api() {
    static CusolverApi api = [] {
        CusolverApi a;
        const char* names[] = {"libcusolver.so.11", "libcusolver.so", "/usr/local/cuda/lib64/libcusolver.so.11"};
        for (const char* nm : names) {
            a.lib = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
            if (a.lib) break;
        }
        if (!a.lib) return a;
#define PIPSORT_SYM(field, name) a.field = reinterpret_cast<decltype(a.field)>(dlsym(a.lib, name))
        PIPSORT_SYM(Create, "cusolverDnCreate");
        PIPSORT_SYM(Destroy, "cusolverDnDestroy");
        PIPSORT_SYM(SetStream, "cusolverDnSetStream");
        PIPSORT_SYM(Dgetrf_bufferSize, "cusolverDnDgetrf_bufferSize");
        PIPSORT_SYM(Dgetrf, "cusolverDnDgetrf");
        PIPSORT_SYM(Dsyevd_bufferSize, "cusolverDnDsyevd_bufferSize");
        PIPSORT_SYM(Dsyevd, "cusolverDnDsyevd");
        PIPSORT_SYM(Dpotrf_bufferSize, "cusolverDnDpotrf_bufferSize");
        PIPSORT_SYM(Dpotrf, "cusolverDnDpotrf");
        PIPSORT_SYM(Dpotrs, "cusolverDnDpotrs");
        a.ok = a.Create && a.Destroy && a.SetStream && a.Dgetrf_bufferSize && a.Dgetrf && a.Dsyevd_bufferSize && a.Dsyevd;
        a.chol = a.Dpotrf_bufferSize && a.Dpotrf && a.Dpotrs;
        return a;
    }();
    return api;
}

// dst (column-major, as cuSOLVER reads it) = the ROW-major src + shift * I: a tiled transpose, so that Dgetrf factorises the
// very matrix gsl_linalg_LU_decomp does (util.cpp:205-214) -- same pivot search per column, same under/overflow pattern of
// the determinant product -- also when the LD file is not exactly symmetric.
__global__ void __launch_bounds__(256) prep_shift_copy_kernel(const double* __restrict__ src, double* __restrict__ dst, int n, double shift) {
    __shared__ double tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int i = by + r, j = bx + threadIdx.x;                 // src row i, column j
        if (i < n && j < n) tile[r][threadIdx.x] = src[(size_t)i * n + j] + (i == j ? shift : 0.0);
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int j = bx + r, i = by + threadIdx.x;                 // dst column-major element (i, j) lives at dst[j * n + i]
        if (i < n && j < n) dst[(size_t)j * n + i] = tile[threadIdx.x][r];
    }
}

// A[i][j] = A[j][i] for j > i (row-major): gsl_eigen_symmv reads the lower triangle only (util.cpp:242), so the matrix
// that is eigen-decomposed -- and with it the effective LD B^T B -- is the symmetric completion of the lower triangle.
__global__ void prep_symmetrise_kernel(double* __restrict__ A, int n) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)n * n) return;
    const size_t i = idx / n, j = idx - i * n;
    if (j > i) A[idx] = A[j * n + i];
}

__global__ void prep_diag_add_kernel(double* __restrict__ A, int n, double shift) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A[(size_t)i * n + i] += shift;
}

// gsl_linalg_LU_det: det = signum * prod_i LU(i,i), multiplied in index order in ONE thread so that the running
// product under/overflows exactly where the reference's does (util.cpp:214-215).  signum from the LAPACK pivots.
__global__ void prep_lu_det_kernel(const double* __restrict__ lu, const int* __restrict__ ipiv, int n, double* __restrict__ det) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    double d = 1.0;
    for (int i = 0; i < n; i++)
        if (ipiv[i] != i + 1) d = -d;
    for (int i = 0; i < n; i++) d *= lu[(size_t)i * n + i];
    *det = d;
}

// t[i] = (q_i . z)^2 / |w_i|   -- one block per eigenvector (column i of the column-major Q)
__global__ void __launch_bounds__(256) prep_k_terms_kernel(const double* __restrict__ Q, const double* __restrict__ w,
                                                           const double* __restrict__ z, int n, double* __restrict__ t) {
    __shared__ double red[256];
    const int i = blockIdx.x;
    const double* q = Q + (size_t)i * n;
    double s = 0.0;
    for (int r = threadIdx.x; r < n; r += 256) s = fma(q[r], z[r], s);
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) t[i] = red[0] * red[0] / fabs(w[i]);
}

// out[0] = sum_i t[i] in a fixed (deterministic) order; out[1] = min |w_i|; out[2] = number of negative eigenvalues
__global__ void __launch_bounds__(256) prep_k_sum_kernel(const double* __restrict__ t, const double* __restrict__ w, int n,
                                                         double* __restrict__ out) {
    __shared__ double red[256], mn[256];
    __shared__ int neg[256];
    double s = 0.0, m = 1.0e300;
    int c = 0;
    for (int r = threadIdx.x; r < n; r += 256) { s += t[r]; m = fmin(m, fabs(w[r])); c += w[r] < 0.0; }
    red[threadIdx.x] = s; mn[threadIdx.x] = m; neg[threadIdx.x] = c;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            red[threadIdx.x] += red[threadIdx.x + o];
            mn[threadIdx.x] = fmin(mn[threadIdx.x], mn[threadIdx.x + o]);
            neg[threadIdx.x] += neg[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) { out[0] = red[0]; out[1] = mn[0]; out[2] = (double)neg[0]; }
}

// out[0] = a . b in a fixed order (one block)
__global__ void __launch_bounds__(256) prep_dot_kernel(const double* __restrict__ a, const double* __restrict__ b, int n, double* __restrict__ out) {
    __shared__ double red[256];
    double s = 0.0;
    for (int r = threadIdx.x; r < n; r += 256) s = fma(a[r], b[r], s);
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = red[0];
}

// A += 2 |w_i| q_i q_i^T for every negative eigenvalue (model.h:227 takes |Omega|)
__global__ void prep_abs_fix_kernel(double* __restrict__ A, const double* __restrict__ Q, const double* __restrict__ w, int n) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)n * n) return;
    const size_t r = idx / n, c = idx - r * n;
    double acc = 0.0;
    for (int i = 0; i < n && w[i] < 0.0; i++)   // Dsyevd returns the eigenvalues in ascending order
        acc = fma(-2.0 * w[i] * Q[(size_t)i * n + r], Q[(size_t)i * n + c], acc);
    A[idx] += acc;
}

// ---- certificates that spare most LU factorizations of the PSD loop -----------------------------------------------------
// util.cpp:204-221 keeps adding 0.01 while the LU determinant -- the product of the pivots in index order -- is not > 0.  For
// thousands of SNPs the product UNDERFLOWS (every pivot < 1), so the loop runs dozens of times although the matrix has long
// been positive definite (it ends when the running product gets stuck at the smallest denormal: every remaining pivot
// > 0.5).  Whether a shift fails can be decided without its LU:
//   * the shifted matrix is symmetric and has a Cholesky factor L (3 ms instead of 24 ms at 5000 SNPs);
//   * every column of L has its largest entry on the diagonal  =>  partial pivoting never swaps rows (the candidates of
//     column k are l_ik l_kk), so the LU pivots ARE l_kk^2 up to rounding;
//   * the running product of the pivots INFLATED by 1e-8 (far more than that rounding) still reaches exactly 0  =>  so
//     does the reference's (rounded multiplication is monotone in each factor).
// A shift without such a certificate gets its real LU, in particular the first one that might pass.
__global__ void prep_is_symmetric_kernel(const double* __restrict__ A, int n, int* __restrict__ asym) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)n * n) return;
    const size_t i = idx / n, j = idx - i * n;
    if (j > i && A[idx] != A[j * n + i]) *asym = 1;
}

// dst = src + shift I (no transpose needed: only called for symmetric matrices)
__global__ void prep_shift_plain_kernel(const double* __restrict__ src, double* __restrict__ dst, int n, double shift) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)n * n) return;
    const size_t i = idx / n, j = idx - i * n;
    dst[idx] = src[idx] + (i == j ? shift : 0.0);
}

// Lf: potrf output, factor in the UPPER triangle of the column-major view (U^T U, U[k][i] at Lf[i * n + k], i >= k), i.e. row k
// of U = column k of L.  One block per k: flag[0] = 1 when some |u_ki| is not clearly below u_kk.
__global__ void __launch_bounds__(256) prep_chol_colmax_kernel(const double* __restrict__ Lf, int n, int* __restrict__ flag) {
    const int k = blockIdx.x;
    const double d = Lf[(size_t)k * n + k] * (1.0 - 1e-8);
    bool bad = !(d > 0.0);
    for (int i = k + 1 + threadIdx.x; i < n; i += 256) bad |= !(fabs(Lf[(size_t)i * n + k]) < d);
    if (bad) *flag = 1;
}

// out[0] = the running product of the inflated pivots u_kk^2 (1 + 1e-8) in index order (one thread, like gsl_linalg_LU_det)
__global__ void prep_chol_product_kernel(const double* __restrict__ Lf, int n, double* __restrict__ out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    double d = 1.0;
    for (int i = 0; i < n; i++) {
        const double u = Lf[(size_t)i * n + i];
        d *= (u * u) * (1.0 + 1e-8);
    }
    out[0] = d;
}

struct PrepResult {
    double add_diag = 0, K = 0, min_abs_eig = 0;
    int n_negative = 0, psd_iterations = 0;
};

// dA: n x n LD on the device, replaced by the effective LD.  dz: n z-scores.  Returns 0, or a negative code:
//  -1 cuSOLVER unavailable, -2 CUDA/cuSOLVER failure, -3 the determinant never became positive.
inline int prep_study_device(cudaStream_t stream, int n, double* dA, const double* dz, PrepResult* res, std::string* why,
                             unsigned long long* launches) {
    *res = PrepResult();
    if (n == 0) return 0;
    const auto t_enter = std::chrono::steady_clock::now();
    const CusolverApi& cs = cusolver_api();
    if (!cs.ok) { *why = "cuSOLVER (libcusolver.so.11) could not be loaded"; return -1; }
    cusolverDnHandle_t h = nullptr;
    if (cs.Create(&h) != CUSOLVER_STATUS_SUCCESS) { *why = "cusolverDnCreate failed"; return -2; }
    auto destroy_handle = scope_exit([&] { cudaStreamSynchronize(stream); cs.Destroy(h); });   // after the buffers below
    DevTemp<double> dW, dwork, dev, dt, dscal;
    DevTemp<int> dipiv, dinfo, dflag;
    const size_t nn = (size_t)n * n;
#define PREP_CU(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { *why = std::string(#call " failed: ") + cudaGetErrorString(e__); return -2; } } while (0)
#define PREP_CS(call) do { cusolverStatus_t s__ = (call); if (s__ != CUSOLVER_STATUS_SUCCESS) { *why = std::string(#call " failed: status ") + std::to_string((int)s__); return -2; } } while (0)
    PREP_CS(cs.SetStream(h, stream));
    int lw_lu = 0, lw_ev = 0;
    PREP_CU(dW.alloc(nn, stream));
    PREP_CU(dev.alloc(n, stream));
    PREP_CU(dt.alloc(n, stream));
    PREP_CU(dscal.alloc(4, stream));
    PREP_CU(dipiv.alloc(n, stream));
    PREP_CU(dinfo.alloc(1, stream));
    PREP_CS(cs.Dgetrf_bufferSize(h, n, n, dW, n, &lw_lu));
    PREP_CS(cs.Dsyevd_bufferSize(h, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_UPPER, n, dW, n, dev, &lw_ev));
    PREP_CU(dwork.alloc(std::max(std::max(lw_lu, lw_ev), 1), stream));
    const unsigned blocks = (unsigned)((nn + 255) / 256);

    static const bool trace = getenv("PIPSORT_TRACE_PREP") != nullptr;
    auto tnow = [&]() { if (trace) cudaStreamSynchronize(stream); return std::chrono::steady_clock::now(); };
    auto tms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::milli>(b - a).count(); };
    const auto t_setup = tnow();
    if (trace) fprintf(stderr, "[prep] n=%d: handle + buffers %.1f ms\n", n, tms(t_enter, t_setup));
    // 1. makeSigmaPositiveSemiDefinite
    double addDiag = 0.0;
    int iters = 0, n_lu = 0, n_cert = 0;
    static const int chol_min = [] { const char* v = getenv("PIPSORT_PREP_CHOL_MIN"); return v ? atoi(v) : 1024; }();
    bool use_chol = cs.chol && n >= chol_min;
    int lw_ch = 0;
    if (use_chol) {
        PREP_CU(dflag.alloc(2, stream));
        PREP_CU(cudaMemsetAsync(dflag, 0, 2 * sizeof(int), stream));
        prep_is_symmetric_kernel<<<blocks, 256, 0, stream>>>(dA, n, dflag);
        int asym = 0;
        PREP_CU(cudaMemcpyAsync(&asym, dflag, sizeof asym, cudaMemcpyDeviceToHost, stream));
        PREP_CU(cudaStreamSynchronize(stream));
        if (asym) use_chol = false;                 // the reference factorises the matrix as read: no certificate for those
        else {
            PREP_CS(cs.Dpotrf_bufferSize(h, CUBLAS_FILL_MODE_UPPER, n, dW, n, &lw_ch));
            if (lw_ch > std::max(std::max(lw_lu, lw_ev), 1)) use_chol = false;   // (never: potrf needs less than getrf / syevd)
        }
    }
    for (;;) {
        bool certified = false;
        if (use_chol) {                             // can this shift be shown to fail without its LU?
            PREP_CU(cudaMemsetAsync(dflag, 0, 2 * sizeof(int), stream));
            prep_shift_plain_kernel<<<blocks, 256, 0, stream>>>(dA, dW, n, addDiag);
            PREP_CS(cs.Dpotrf(h, CUBLAS_FILL_MODE_UPPER, n, dW, n, dwork, lw_ch, dinfo));
            prep_chol_colmax_kernel<<<n, 256, 0, stream>>>(dW, n, dflag);
            prep_chol_product_kernel<<<1, 32, 0, stream>>>(dW, n, dscal);
            *launches += 3;
            int hinfo = 0, hflag[2] = {0, 0};
            double prod = 1.0;
            PREP_CU(cudaMemcpyAsync(&hinfo, dinfo, sizeof hinfo, cudaMemcpyDeviceToHost, stream));
            PREP_CU(cudaMemcpyAsync(hflag, dflag, sizeof hflag, cudaMemcpyDeviceToHost, stream));
            PREP_CU(cudaMemcpyAsync(&prod, dscal, sizeof prod, cudaMemcpyDeviceToHost, stream));
            PREP_CU(cudaStreamSynchronize(stream));
            certified = hinfo == 0 && hflag[0] == 0 && prod == 0.0;
        }
        if (certified) {
            n_cert++;
        } else {
            prep_shift_copy_kernel<<<dim3((n + 31) / 32, (n + 31) / 32), dim3(32, 8), 0, stream>>>(dA, dW, n, addDiag);
            PREP_CS(cs.Dgetrf(h, n, n, dW, n, dwork, dipiv, dinfo));
            prep_lu_det_kernel<<<1, 32, 0, stream>>>(dW, dipiv, n, dscal);
            *launches += 2;
            n_lu++;
            double det = 0.0;
            PREP_CU(cudaMemcpyAsync(&det, dscal, sizeof det, cudaMemcpyDeviceToHost, stream));
            PREP_CU(cudaStreamSynchronize(stream));
            if (det > 0) { iters++; break; }
        }
        iters++;
        addDiag += 0.01;                        // accumulated exactly like util.cpp:219
        if (iters > 100000) { *why = "the LD matrix never reached a positive determinant"; return -3; }
    }
    const auto t_psd = tnow();
    if (trace) fprintf(stderr, "[prep] PSD loop: %d shifts (%d LU factorizations, %d Cholesky certificates) %.1f ms (shift %.2f)\n", iters,
                       n_lu, n_cert, tms(t_setup, t_psd), addDiag);
    // 2. eigen-decomposition of Sigma + a I  (GSL reads the lower triangle of the row-major matrix = the upper
    //    triangle of the column-major view)
    prep_diag_add_kernel<<<(n + 255) / 256, 256, 0, stream>>>(dA, n, addDiag);
    prep_symmetrise_kernel<<<blocks, 256, 0, stream>>>(dA, n);
    *launches += 2;
    PREP_CU(cudaMemcpyAsync(dW, dA, nn * sizeof(double), cudaMemcpyDeviceToDevice, stream));
    if (use_chol) {
        // positive definite after the shift (the usual case): Omega > 0, so B^T B is the matrix itself and
        // K = S'^T S' = z^T (Sigma + a I)^-1 z -- one Cholesky solve instead of the eigen-decomposition
        PREP_CS(cs.Dpotrf(h, CUBLAS_FILL_MODE_UPPER, n, dW, n, dwork, lw_ch, dinfo));
        int hinfo = 0;
        PREP_CU(cudaMemcpyAsync(&hinfo, dinfo, sizeof hinfo, cudaMemcpyDeviceToHost, stream));
        PREP_CU(cudaStreamSynchronize(stream));
        if (hinfo == 0) {
            PREP_CU(cudaMemcpyAsync(dt, dz, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, stream));
            PREP_CS(cs.Dpotrs(h, CUBLAS_FILL_MODE_UPPER, n, 1, dW, n, dt, n, dinfo));
            prep_dot_kernel<<<1, 256, 0, stream>>>(dz, dt, n, dscal);
            *launches += 1;
            double Kc = 0.0;
            PREP_CU(cudaMemcpyAsync(&Kc, dscal, sizeof Kc, cudaMemcpyDeviceToHost, stream));
            PREP_CU(cudaStreamSynchronize(stream));
            if (trace) fprintf(stderr, "[prep] positive definite: K by Cholesky solve %.1f ms\n", tms(t_psd, tnow()));
            res->add_diag = addDiag; res->K = Kc; res->min_abs_eig = 0.0; res->n_negative = 0; res->psd_iterations = iters;
            return 0;
        }
        PREP_CU(cudaMemcpyAsync(dW, dA, nn * sizeof(double), cudaMemcpyDeviceToDevice, stream));   // not definite: the eigen path
    }
    PREP_CS(cs.Dsyevd(h, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_UPPER, n, dW, n, dev, dwork, std::max(lw_ev, 1), dinfo));
    int info = 0;
    PREP_CU(cudaMemcpyAsync(&info, dinfo, sizeof info, cudaMemcpyDeviceToHost, stream));
    // 3. K and the |Omega| correction
    prep_k_terms_kernel<<<n, 256, 0, stream>>>(dW, dev, dz, n, dt);
    prep_k_sum_kernel<<<1, 256, 0, stream>>>(dt, dev, n, dscal);
    *launches += 3;
    double sc[3] = {0, 0, 0};
    PREP_CU(cudaMemcpyAsync(sc, dscal, sizeof sc, cudaMemcpyDeviceToHost, stream));
    PREP_CU(cudaStreamSynchronize(stream));
    if (trace) fprintf(stderr, "[prep] eigen-decomposition + K: %.1f ms\n", tms(t_psd, tnow()));
    if (info != 0) { *why = "cusolverDnDsyevd did not converge (info " + std::to_string(info) + ")"; return -2; }
    if (sc[2] > 0) {
        prep_abs_fix_kernel<<<blocks, 256, 0, stream>>>(dA, dW, dev, n);
        *launches += 1;
    }
    PREP_CU(cudaGetLastError());
    res->add_diag = addDiag; res->K = sc[0]; res->min_abs_eig = sc[1]; res->n_negative = (int)sc[2]; res->psd_iterations = iters;
#undef PREP_CU
#undef PREP_CS
    return 0;
}

}  // namespace pipsort
