// Optimal Kronecker-factored variational covariance of the B1 (ASVGP) and VGGP_SVGP_MARKOV families (DESIGN.md section 4,
// K1s): one coordinate update of S_d = tril(L_d) tril(L_d)^T with theta, m and every S_e, e != d, fixed.
//
// With s = ell_scale, the S_d-dependent part of the ELBO is -(1/2) tr(S_d A_d) + (M / (2 M_d)) log det S_d, maximised by
// S_d = (M / M_d) A_d^-1.  In both families A_d comes from one tridiagonal matrix
//     T_d = (s / noise) H_d + c_d F_d,   H_d = sum_n (prod_{e != d} q_e(x_n)) w_d w_d^T   (the gbuf band [bq_diag | bq_off]),
//                                        c_d = prod_{e != d} tr(K_e^-1 S_e)                (plan scalars of the last forward)
//     Markov:  F_d = K_d^-1,  A_d = T_d,              S_d = (M / M_d) T_d^-1
//     B1:      F_d = K_d,     A_d = P_d T_d P_d,      S_d = (M / M_d) K_d T_d^-1 K_d     (P_d = K_d^-1)
// T_d = U U^T with U upper bidiagonal (UL factorisation, backward recurrence), so T_d^-1 = U^-T U^-1 and
//     Markov:  L_d = sqrt(M / M_d) U^-T                               (lower triangular, positive diagonal)
//     B1:      X = sqrt(M / M_d) K_d U^-T is lower Hessenberg; X X^T = S_d, and an RQ sweep of Givens rotations over
//              neighbouring columns (X = L Q) leaves the Cholesky factor L_d.
// Column j of U^-T solves U^T y = e_j: y_j = 1 / b_j, y_k = -(e_k / b_k) y_{k-1} (b: diagonal of U, e_k = U[k-1][k]); the
// magnitudes only decay down a column, so the recurrence is stable.
//
// Storage: the only M_d^2 memory is the caller's output block.  The B1 sweep keeps X's strictly lower part transposed in
// the strict upper triangle of that block and its diagonal and superdiagonal in O(M_d) scratch, so the lower triangle
// still holds the old factor until the thread that owns a row overwrites an entry with its final value.  That thread reads
// the old entry first, which makes the change measure work when the output aliases the input.
//
// Change measure: ||L_new / ||L_new|| - L_old / ||L_old|| ||_F (lower triangles), invariant under S_1 -> a S_1,
// S_2 -> S_2 / a.  With d = L_new - L_old, a = ||L_new||, b = ||L_old||:  L_new / a - L_old / b = d / a + L_old (b - a) / (a b),
// so its square is  sum d^2 / a^2 + 2 (b - a) sum(d L_old) / (a^2 b) + (b - a)^2 / a^2  with b - a = sum(-d (L_new + L_old)) / (a + b):
// four sums, no cancellation between nearly equal norms.
#pragma once
#include "grid.cuh"
#include "svgpm.cuh"

namespace vggp {

constexpr int CO_THREADS = 256;      // threads of the factor and sweep CTAs and of the column kernels
constexpr int CO_ROWS = 10;          // rows per thread of the sweep
constexpr int CO_MAX_N = CO_THREADS * CO_ROWS;     // 2560, the largest B1 dimension; T_d is staged in 40 KB of shared memory

// scratch (float64, 6 n + 8): F band [fd | fo], U^-T recurrence [ib = 1 / b_k | rr = -e_k / b_k], B1 X [xd | xs], the four
// change sums, the status (0 ok, 1 failed pivot)
struct CoArgs {
    int n, d, D, family;
    double scale;                    // sqrt(M / M_d)
    double* fd; double* fo;          // F_d band: diag, off (F[k][k+1])
    double* ib; double* rr;
    double* xd; double* xs;          // B1: X[k][k], X[k][k+1]
    double* acc;                     // [sum new^2, sum old^2, sum d^2, sum d old] then the status
    const double* Lold;              // block d of the input
    double* Lout;                    // block d of the output
};

__device__ __forceinline__ bool co_failed(const CoArgs& a) { return a.acc[4] != 0.0; }

// one CTA: F_d band, T_d, its UL factorisation.  `band`: [bp_diag | bp_off | bq_diag | bq_off] of dimension d (obs dtype).
template <typename T>
__global__ void __launch_bounds__(CO_THREADS) k_co_factor(CoArgs a, const __grid_constant__ GridDims g,
                                                          const double* __restrict__ svw, const T* __restrict__ band,
                                                          const double* __restrict__ theta, const double* __restrict__ trs,
                                                          double ell_scale, int* __restrict__ info) {
    const int n = a.n, d = a.d;
    double c = 1.0;
    for (int e = 0; e < a.D; ++e)
        if (e != d) c *= trs[e];
    const double cs = ell_scale / theta[2 * a.D];
    __shared__ double td[CO_MAX_N], to[CO_MAX_N];
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double fd, fo;
        if (a.family == VGGP_B1_ASVGP) {
            fd = factor_entry(g, theta, d, i, i);
            fo = i + 1 < n ? factor_entry(g, theta, d, i, i + 1) : 0.0;
        } else {
            fd = svw[SVW_PD * n + i];
            fo = i + 1 < n ? svw[SVW_PO * n + i] : 0.0;
        }
        a.fd[i] = fd;
        a.fo[i] = fo;
        td[i] = cs * (double)band[2 * n + i] + c * fd;                               // T[i][i]
        to[i] = i + 1 < n ? cs * (double)band[3 * n + i] + c * fo : 0.0;            // T[i][i+1]
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    // T = U U^T:  b_k^2 = T[k][k] - e_{k+1}^2,  e_k = T[k-1][k] / b_k
    double e = 0.0;
    bool bad = false;
    for (int k = n - 1; k >= 0; --k) {
        const double piv = td[k] - e * e;
        if (!(piv > 0.0) || !isfinite(piv)) { bad = true; break; }
        const double rb = rsqrt(piv);                 // 1 / b_k
        e = k > 0 ? to[k - 1] * rb : 0.0;
        a.ib[k] = rb;
        a.rr[k] = -e * rb;
    }
    for (int k = 0; k < 4; ++k) a.acc[k] = 0.0;
    a.acc[4] = bad ? 1.0 : 0.0;
    if (bad) atomicMax(info, d + 1);
}

__device__ __forceinline__ void co_block_acc(const CoArgs& a, double (&s)[4]) {
    __shared__ double red[32];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double v = block_sum(s[k], red);
        if (threadIdx.x == 0) atomicAdd(a.acc + k, v);
    }
}

__device__ __forceinline__ void co_pair(double nv, double ov, double (&s)[4]) {
    const double df = nv - ov;
    s[0] = fma(nv, nv, s[0]);
    s[1] = fma(ov, ov, s[1]);
    s[2] = fma(df, df, s[2]);
    s[3] = fma(df, ov, s[3]);
}

// Markov: L_out = scale U^-T, thread j owns column j and walks every row, so the writes of a row are consecutive.
__global__ void __launch_bounds__(CO_THREADS) k_co_markov(CoArgs a) {
    if (co_failed(a)) return;
    const int n = a.n, j = (int)blockIdx.x * blockDim.x + threadIdx.x;
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    if (j < n) {
        double x = a.scale * a.ib[j];
        for (int k = 0; k < n; ++k) {
            const i64 o = (i64)k * n + j;
            if (k < j) { a.Lout[o] = 0.0; continue; }
            if (k > j) x *= a.rr[k];
            co_pair(x, a.Lold[o], s);
            a.Lout[o] = x;
        }
    }
    co_block_acc(a, s);
}

// B1: column j of X = scale K_d U^-T.  X[j-1][j] -> xs[j-1], X[j][j] -> xd[j], X[k][j] (k > j) -> L_out[j][k].
__global__ void __launch_bounds__(CO_THREADS) k_co_b1_x(CoArgs a) {
    if (co_failed(a)) return;
    const int n = a.n, j = (int)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    double yp = 0.0, yc = a.ib[j];                        // y[k-1], y[k] at k = j
    if (j > 0) a.xs[j - 1] = a.scale * a.fo[j - 1] * yc;
    for (int k = j; k < n; ++k) {
        const double yn = k + 1 < n ? a.rr[k + 1] * yc : 0.0;
        const double v = a.scale * ((k > 0 ? a.fo[k - 1] * yp : 0.0) + a.fd[k] * yc + a.fo[k] * yn);
        if (k == j) a.xd[j] = v;
        else a.Lout[(i64)j * n + k] = v;
        yp = yc;
        yc = yn;
    }
    if (j == n - 1) a.xs[n - 1] = 0.0;
}

// B1: RQ sweep X = L Q, one CTA.  Row r = threadIdx.x + i CO_THREADS carries its current column-k entry; at step k the owner
// of row k builds the rotation of columns k, k+1 that zeroes X[k][k+1], every row below applies it and stores its final
// L[r][k].  The original X[r][k+1] and the old L[r][k] do not depend on the rotations and are loaded one step ahead, also
// by the row that owns the next step, so that no global load sits on the chain of steps.
__global__ void __launch_bounds__(CO_THREADS) k_co_b1_rq(CoArgs a) {
    if (co_failed(a)) return;
    __shared__ double rot[2][2];
    const int n = a.n, t = threadIdx.x;
    double carry[CO_ROWS], nx[CO_ROWS], no[CO_ROWS];
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    // X[r][c] for c <= r + 1 (the caller guarantees c <= r + 1)
    auto xat = [&](int r, int c) -> double {
        if (c == r) return a.xd[r];
        if (c == r + 1) return a.xs[r];
        return a.Lout[(i64)c * n + r];
    };
#pragma unroll
    for (int i = 0; i < CO_ROWS; ++i) {
        const int r = t + i * CO_THREADS;
        carry[i] = 0.0; nx[i] = 0.0; no[i] = 0.0;
        if (r < n) {
            carry[i] = xat(r, 0);
            nx[i] = xat(r, 1);
            no[i] = a.Lold[(i64)r * n];
        }
    }
    for (int k = 0; k < n - 1; ++k) {
        double xk1[CO_ROWS], ok[CO_ROWS];
#pragma unroll
        for (int i = 0; i < CO_ROWS; ++i) {          // values of this step, prefetch of the next
            const int r = t + i * CO_THREADS;
            xk1[i] = nx[i];
            ok[i] = no[i];
            if (r < n && r >= k + 1) {
                nx[i] = xat(r, k + 2);
                no[i] = a.Lold[(i64)r * n + k + 1];
            }
        }
        if ((k & (CO_THREADS - 1)) == t) {
            const int i = k / CO_THREADS;
            double cv = 0.0, b = 0.0, od = 0.0;
#pragma unroll
            for (int q = 0; q < CO_ROWS; ++q)
                if (q == i) { cv = carry[q]; b = xk1[q]; od = ok[q]; }
            const double rho = sqrt(fma(cv, cv, b * b));
            double c = 1.0, sn = 0.0;
            if (rho > 0.0) { const double ir = 1.0 / rho; c = cv * ir; sn = b * ir; }
            rot[k & 1][0] = c;
            rot[k & 1][1] = sn;
            co_pair(rho, od, s);
            a.Lout[(i64)k * n + k] = rho;
        }
        __syncthreads();
        const double c = rot[k & 1][0], sn = rot[k & 1][1];
#pragma unroll
        for (int i = 0; i < CO_ROWS; ++i) {
            const int r = t + i * CO_THREADS;
            if (r < n && r > k) {
                const double v = carry[i], w = xk1[i];
                const double lk = c * v + sn * w;
                carry[i] = c * w - sn * v;
                co_pair(lk, ok[i], s);
                a.Lout[(i64)r * n + k] = lk;
            }
        }
    }
    // last diagonal entry (the rotations leave every other diagonal entry >= 0), then the strict upper triangle
    if (((n - 1) & (CO_THREADS - 1)) == t) {
        const int i = (n - 1) / CO_THREADS;
        double cv = 0.0;
#pragma unroll
        for (int q = 0; q < CO_ROWS; ++q) if (q == i) cv = carry[q];
        cv = fabs(cv);
        co_pair(cv, a.Lold[(i64)(n - 1) * n + n - 1], s);
        a.Lout[(i64)(n - 1) * n + n - 1] = cv;
    }
    __syncthreads();
    for (i64 e = t; e < (i64)n * n; e += CO_THREADS)
        if (e % n > e / n) a.Lout[e] = 0.0;
    co_block_acc(a, s);
}

// change += ||L_new / ||L_new|| - L_old / ||L_old|| ||_F from the four sums (+inf after a failed pivot)
__global__ void k_co_change(const double* __restrict__ acc, double* __restrict__ change) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (acc[4] != 0.0) { *change += INFINITY; return; }
    const double nn = acc[0], oo = acc[1], dd = acc[2], dold = acc[3];
    const double a = sqrt(nn), b = sqrt(oo);
    double v;
    if (!(b > 0.0)) v = 1.0;                      // no previous factor: the whole unit-norm factor is new
    else {
        const double bma = -(dd + 2.0 * dold) / (a + b);    // b - a = sum(-d (L_new + L_old)) / (a + b), L_new + L_old = d + 2 L_old
        v = dd / (a * a) + 2.0 * bma * dold / (a * a * b) + bma * bma / (a * a);
        v = sqrt(fmax(v, 0.0));
    }
    *change += v;
}

}  // namespace vggp
