// Lawson-Hanson non-negative least squares against the handle's X (prmf_nnls_x): the solver behind the pathway-seeded
// initialisation of the reference CLI (script/prmf_runner.py:272-334, :1023-1064), which calls scipy.optimize.nnls
// twice per init pathway, once with A = X^T and once with A = X.
//
// k independent problems x_c = argmin_{x >= 0} ||A x - b_c|| share A.  One outer iteration for all of them:
//   nnls_resid_kernel   r_c = b_c - sum_{j in P_c} x_j a_j   (gathers the few passive columns; written into the W
//                                                             operand of an X stream)
//   X stream + sum      w_c = A^T r_c                        (the pass-1 / pass-2 products of the inner step)
//   nnls_step_kernel    one CTA per problem: entering variable, Gram column, Cholesky row, step back to the boundary
//   nnls_rnorm_kernel   ||r_c|| once the loop has ended
// Column j of A is a contiguous row of X (A = X^T) or of its transposed copy (A = X).  The passive system is solved on
// the normal equations, in the order the columns entered, with a Cholesky factor grown one row per entering column.
// Every reduction runs in a fixed order, so repeated calls give bitwise-identical results.
#pragma once

#include <cfloat>
#include <cstdint>

namespace prmf {

constexpr int kNnlsThreads = 256;
constexpr int kNnlsMaxPassive = 1024;     // passive-set capacity of the workspace (Gram + factor: 16 MB per problem)

// status words
constexpr int kNnlsRunning = 0;
constexpr int kNnlsConverged = 1;
constexpr int kNnlsMaxIter = -1;
constexpr int kNnlsCapacity = -2;
constexpr int kNnlsSingular = -3;

// Per-problem state in one workspace (cap = passive capacity, nun = number of unknowns).  T: element type of the stored
// X (double, or float for PRMF_X_F32 handles, whose values are widened exactly before any arithmetic).
template <typename T>
struct NnlsWork {
    int k = 0, cap = 0;
    int64_t neq = 0, nun = 0;
    const T* Arows = nullptr;                 // column j of A = Arows[j * lda .. + neq)
    int64_t lda = 0;
    const double* Bt = nullptr;               // [k][neq]
    double* w = nullptr;                      // duals [nun][k] (sum of the X-stream partials)
    double* G = nullptr;                      // [k][cap][cap] Gram of the passive columns, lower triangle, entry order
    double* L = nullptr;                      // [k][cap][cap] its Cholesky factor
    double* atb = nullptr;                    // [k][cap] a_j^T b of the passive columns
    double* xP = nullptr;                     // [k][cap] passive coefficients
    int* pidx = nullptr;                      // [k][cap] passive column indices, entry order
    int8_t* flag = nullptr;                   // [k][nun] 0 at its bound, 1 passive, 2 rejected in this round
    int* np = nullptr;                        // [k] passive-set size
    int* iter = nullptr;                      // [k] iterations counted as scipy counts them
    int* status = nullptr;                    // [k]
    double tol = 0.0;
    int maxiter = 0;
};

__device__ __forceinline__ double nnls_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// r[e][c] = b_c[e] - sum_q xP[q] a_{pidx[q]}[e] for the running problems (every problem when `all`), 0 otherwise.
// grid (ceil(neq / 256), k); W has row pitch k.
template <typename T>
__global__ void __launch_bounds__(kNnlsThreads) nnls_resid_kernel(NnlsWork<T> wk, double* __restrict__ W, int all) {
    const int c = blockIdx.y;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= wk.neq) return;
    double r = 0.0;
    if (all || wk.status[c] == kNnlsRunning) {
        r = wk.Bt[(int64_t)c * wk.neq + e];
        const int p = wk.np[c];
        const int* pidx = wk.pidx + (int64_t)c * wk.cap;
        const double* xP = wk.xP + (int64_t)c * wk.cap;
        for (int q = 0; q < p; ++q) r = fma(-xP[q], (double)wk.Arows[(int64_t)pidx[q] * wk.lda + e], r);
    }
    W[e * wk.k + c] = r;
}

// rnorm[c] = ||W[:, c]||, one CTA per problem
__global__ void __launch_bounds__(kNnlsThreads) nnls_rnorm_kernel(const double* __restrict__ W, int64_t neq, int k,
                                                                  double* __restrict__ rnorm) {
    __shared__ double part[kNnlsThreads / 32];
    const int c = blockIdx.x;
    double s = 0.0;
    for (int64_t e = threadIdx.x; e < neq; e += blockDim.x) {
        const double v = W[e * k + c];
        s = fma(v, v, s);
    }
    s = nnls_warp_sum(s);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < kNnlsThreads / 32; ++i) t += part[i];
        rnorm[c] = sqrt(t);
    }
}

// Row i of the Cholesky factor from the Gram row g[0..i] (warp-wide, lanes over the inner sums):
// L[i][t] = (g[t] - sum_{u<t} L[i][u] L[t][u]) / L[t][t], returns the pivot d = g[i] - sum_u L[i][u]^2.
// The row is built in `row` (shared) and is not stored.
__device__ double nnls_chol_row(const double* __restrict__ L, int cap, const double* g, int i, double* row) {
    const int lane = threadIdx.x & 31;
    for (int t = 0; t < i; ++t) {
        const double* Lt = L + (int64_t)t * cap;
        double s = 0.0;
        for (int u = lane; u < t; u += 32) s = fma(row[u], Lt[u], s);
        s = nnls_warp_sum(s);
        if (lane == 0) row[t] = (g[t] - s) / Lt[t];
        __syncwarp();
    }
    double s = 0.0;
    for (int u = lane; u < i; u += 32) s = fma(row[u], row[u], s);
    s = nnls_warp_sum(s);
    return g[i] - s;
}

// s = G^{-1} atb on the first p passive columns through L (warp-wide)
__device__ void nnls_solve(const double* __restrict__ L, int cap, const double* __restrict__ atb, int p,
                           double* y, double* s) {
    const int lane = threadIdx.x & 31;
    for (int i = 0; i < p; ++i) {                       // forward: L y = atb
        const double* Li = L + (int64_t)i * cap;
        double a = 0.0;
        for (int t = lane; t < i; t += 32) a = fma(Li[t], y[t], a);
        a = nnls_warp_sum(a);
        if (lane == 0) y[i] = (atb[i] - a) / Li[i];
        __syncwarp();
    }
    for (int i = p - 1; i >= 0; --i) {                  // backward: L^T s = y
        double a = 0.0;
        for (int t = i + 1 + lane; t < p; t += 32) a = fma(L[(int64_t)t * cap + i], s[t], a);
        a = nnls_warp_sum(a);
        if (lane == 0) s[i] = (y[i] - a) / L[(int64_t)i * cap + i];
        __syncwarp();
    }
}

// a . b over n entries, lanes strided by 32 (widened to fp64 first), summed over the warp
template <typename A, typename B>
__device__ __forceinline__ double nnls_dot(const A* a, const B* b, int64_t n, int lane) {
    double s = 0.0;
    for (int64_t e = lane; e < n; e += 32) s = fma((double)a[e], (double)b[e], s);
    return nnls_warp_sum(s);
}

// (value, index) maximum with the first index winning ties
__device__ __forceinline__ void nnls_argmax_merge(double& v, int& j, double v2, int j2) {
    if (j2 >= 0 && (j < 0 || v2 > v || (v2 == v && j2 < j))) { v = v2; j = j2; }
}

// One outer Lawson-Hanson iteration per running problem, with the duals w of the current x.  The rules are those of
// cv_nnls_kernel (cv.cu) and scipy.optimize.nnls: the entering variable is the largest dual above tol (first index on a
// tie); a candidate whose column is numerically dependent on the passive ones is skipped for the next largest dual; a
// passive coefficient that turns non-positive makes the step stop at the boundary and drops it.  Iterations are counted
// as scipy counts them: one per outer iteration (including the one that finds the optimum) and one per step back.
// The loop also ends when the passive set reaches the number of equations, as the Fortran original does.
template <typename T>
__global__ void __launch_bounds__(kNnlsThreads) nnls_step_kernel(NnlsWork<T> wk) {
    __shared__ double g[kNnlsMaxPassive + 2];
    __shared__ double row[kNnlsMaxPassive];
    __shared__ double y[kNnlsMaxPassive];
    __shared__ double s[kNnlsMaxPassive];
    __shared__ int kept[kNnlsMaxPassive];
    __shared__ double red_v[kNnlsThreads / 32];
    __shared__ int red_j[kNnlsThreads / 32];
    __shared__ int sh_enter, sh_done, sh_nrej;

    const int c = blockIdx.x;
    if (wk.status[c] != kNnlsRunning) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cap = wk.cap;
    const int64_t nun = wk.nun, neq = wk.neq;
    double* G = wk.G + (int64_t)c * cap * cap;
    double* L = wk.L + (int64_t)c * cap * cap;
    double* atb = wk.atb + (int64_t)c * cap;
    double* xP = wk.xP + (int64_t)c * cap;
    int* pidx = wk.pidx + (int64_t)c * cap;
    int8_t* flag = wk.flag + (int64_t)c * nun;
    const double* bc = wk.Bt + (int64_t)c * neq;
    int p = wk.np[c];
    int iter = wk.iter[c] + 1;
    int st = kNnlsRunning;
    if (tid == 0) sh_nrej = 0;
    __syncthreads();

    if (iter > wk.maxiter) st = kNnlsMaxIter;
    while (st == kNnlsRunning) {
        if ((int64_t)p >= nun || (int64_t)p >= neq) { st = kNnlsConverged; break; }
        // entering variable: largest dual among the columns at their bound
        double bv = 0.0;
        int bj = -1;
        for (int64_t j = tid; j < nun; j += blockDim.x)
            if (flag[j] == 0) nnls_argmax_merge(bv, bj, wk.w[j * wk.k + c], (int)j);
        for (int o = 16; o > 0; o >>= 1) {
            const double v2 = __shfl_xor_sync(0xffffffffu, bv, o);
            const int j2 = __shfl_xor_sync(0xffffffffu, bj, o);
            nnls_argmax_merge(bv, bj, v2, j2);
        }
        if (lane == 0) { red_v[warp] = bv; red_j[warp] = bj; }
        __syncthreads();
        if (tid == 0) {
            double v = 0.0;
            int j = -1;
            for (int i = 0; i < kNnlsThreads / 32; ++i) nnls_argmax_merge(v, j, red_v[i], red_j[i]);
            sh_enter = (j >= 0 && v > wk.tol) ? j : -1;
        }
        __syncthreads();
        const int enter = sh_enter;
        if (enter < 0) { st = kNnlsConverged; break; }
        if (p >= cap) { st = kNnlsCapacity; break; }
        // Gram column of the candidate: a_enter . a_i (i passive), a_enter . a_enter, a_enter . b -- a warp per dot
        const T* aj = wk.Arows + (int64_t)enter * wk.lda;
        for (int q = warp; q < p + 2; q += kNnlsThreads / 32) {
            double a;
            if constexpr (sizeof(T) == sizeof(double)) {
                const double* other = q < p ? wk.Arows + (int64_t)pidx[q] * wk.lda : q == p ? aj : bc;
                a = nnls_dot(aj, other, neq, lane);
            } else {                                         // b is fp64, the columns of A are not
                a = q <= p ? nnls_dot(aj, q < p ? wk.Arows + (int64_t)pidx[q] * wk.lda : aj, neq, lane)
                           : nnls_dot(aj, bc, neq, lane);
            }
            if (lane == 0) g[q] = a;
        }
        __syncthreads();
        if (warp == 0) {
            const double d = nnls_chol_row(L, cap, g, p, row);
            if (lane == 0) {
                // Lawson & Hanson's independence test: a column that is (nearly) a combination of the passive ones
                // cannot lower the residual -- leave it at zero for this round and try the next largest dual
                if (!(d > 1e-13 * g[p])) {
                    flag[enter] = 2;
                    ++sh_nrej;
                    sh_done = 0;
                } else {
                    double* Gp = G + (int64_t)p * cap;
                    double* Lp = L + (int64_t)p * cap;
                    for (int t = 0; t <= p; ++t) Gp[t] = g[t];
                    for (int t = 0; t < p; ++t) Lp[t] = row[t];
                    Lp[p] = sqrt(d);
                    atb[p] = g[p + 1];
                    xP[p] = 0.0;
                    pidx[p] = enter;
                    flag[enter] = 1;
                    sh_done = 1;
                }
            }
        }
        __syncthreads();
        if (!sh_done) continue;
        ++p;
        if (sh_nrej) {
            for (int64_t j = tid; j < nun; j += blockDim.x)
                if (flag[j] == 2) flag[j] = 0;
            __syncthreads();
            if (tid == 0) sh_nrej = 0;
        }
        // the passive system, then back along the segment while a coefficient is not positive
        if (warp == 0) {
            __syncwarp();
            nnls_solve(L, cap, atb, p, y, s);
            while (true) {
                bool neg = false;
                for (int q = lane; q < p; q += 32) neg |= s[q] < 0.0;
                if (!__any_sync(0xffffffffu, neg)) break;
                if (++iter > wk.maxiter) { st = kNnlsMaxIter; break; }
                double alpha = DBL_MAX;
                for (int q = lane; q < p; q += 32)
                    if (s[q] < 0.0) alpha = fmin(alpha, xP[q] / (xP[q] - s[q]));
                for (int o = 16; o > 0; o >>= 1) alpha = fmin(alpha, __shfl_xor_sync(0xffffffffu, alpha, o));
                for (int q = lane; q < p; q += 32) xP[q] = xP[q] * (1.0 - alpha) + alpha * s[q];
                __syncwarp();
                // drop the coefficients that reached the bound; keep the entry order of the others
                int np_ = 0, first = p;
                if (lane == 0) {
                    for (int q = 0; q < p; ++q) {
                        if (xP[q] <= wk.tol) { flag[pidx[q]] = 0; if (first == p) first = q; }
                        else kept[np_++] = q;
                    }
                }
                np_ = __shfl_sync(0xffffffffu, np_, 0);
                first = __shfl_sync(0xffffffffu, first, 0);
                __syncwarp();
                for (int a = first; a < np_; ++a) {      // kept[a] > a for a >= first: rows move up in place
                    const int src = kept[a];
                    const double* Gs = G + (int64_t)src * cap;
                    double* Ga = G + (int64_t)a * cap;
                    for (int b = lane; b <= a; b += 32) {
                        const int sb = kept[b];
                        Ga[b] = Gs[sb];
                    }
                    if (lane == 0) { atb[a] = atb[src]; xP[a] = xP[src]; pidx[a] = pidx[src]; }
                    __syncwarp();
                }
                p = np_;
                bool ok = true;
                for (int i = first; i < p && ok; ++i) {   // the factor rows from the first dropped column on
                    const double* Gi = G + (int64_t)i * cap;
                    const double d = nnls_chol_row(L, cap, Gi, i, row);
                    ok = d > 1e-13 * Gi[i];
                    if (ok) {
                        double* Li = L + (int64_t)i * cap;
                        for (int t = lane; t < i; t += 32) Li[t] = row[t];
                        if (lane == 0) Li[i] = sqrt(d);
                    }
                    __syncwarp();
                }
                if (!ok) { st = kNnlsSingular; break; }
                nnls_solve(L, cap, atb, p, y, s);
            }
            if (st == kNnlsRunning)
                for (int q = lane; q < p; q += 32) xP[q] = s[q];
        }
        break;   // x changed: its duals need another pass over X
    }
    __syncthreads();
    if (tid == 0) {
        wk.np[c] = p;
        wk.iter[c] = iter;
        wk.status[c] = st;
    }
}

}  // namespace prmf
