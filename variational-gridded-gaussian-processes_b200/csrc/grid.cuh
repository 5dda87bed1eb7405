// Dense grid side of the B0, SVGP and VFF families: per-dimension factor build, blocked Cholesky, triangular inverse
// leaves, band / trace / log-det reductions, and the elementwise + reduction pieces of the reverse pass.  All float64.
// The entries of every family's factor K_d (factor_entry, factor_entry_grad) are shared with the fused B1 grid side
// (grid_b1.cuh), the optimal mean (meanopt.cuh) and the optimal covariance (covopt.cuh).
// Maths: SURVEY.md appendix A.  Reference formulas: gridded_kronecker_structure.py:731-780 (B1/ASVGP Kuu),
// :1286-1323 (B0 Toeplitz Kuu).
#pragma once
#include "common.cuh"

namespace vggp {

constexpr int NB = 64;            // Cholesky / triangular-inverse block size
constexpr int MAX_LEAVES = 40;    // supports M_d <= 2560

// scalar slots in the plan's float64 scalar block
enum {
    SC_LOGDETK = 0,   // [3]
    SC_LOGDETS = 3,   // [3]
    SC_TR = 6,        // [3] tr(P_d S_d)
    SC_MALPHA = 9,    // <m, alpha>
    SC_COUNT = 16
};

struct GridDims {
    int D, family, obs_dtype;
    int n[VGGP_MAX_D];            // M_d
    int K[VGGP_MAX_D];            // knots
    float delta32[VGGP_MAX_D];    // mesh[1] - mesh[0] in float32 (reference: SplineBasis.delta, bspline.py:89)
    const float* knots[VGGP_MAX_D];   // device copy of the knots (SVGP family: the inducing locations z_i)
    i64 M;
    i64 Loff[VGGP_MAX_D];         // offset of L_d inside the concatenated L / dL arrays
    int band_off[VGGP_MAX_D];     // offset (elements) of dim d's block inside the gbuf band part [bp_d|bp_o|bq_d|bq_o]
    int tab_off[VGGP_MAX_D];      // offset (elements) of dim d's block inside the per-cell tables (8 n_d each)
    i64 gfac_off[VGGP_MAX_D];     // B0 family: offset of dim d's [bP | bQ] block inside the gbuf factor part
    // allocated by every plan but the Markov SVGP's: K_d as built and P_d = K_d^-1 (B1: filled on demand by
    // vggp_workspace_ptr), R_d = P_d tril(L_d), the band of Q_d = R_d R_d^T
    double* Kraw[VGGP_MAX_D];
    double* P[VGGP_MAX_D];
    double* R[VGGP_MAX_D];
    double* Qb[VGGP_MAX_D];       // float64 main / first off diagonal of Q_d: [diag (n) | off (n)]
    // allocated by the dense families only (B0, SVGP, VFF): the blocked Cholesky, triangular inverse and GEMM products
    double* cdiag[VGGP_MAX_D];    // NB x NB: factored diagonal block of the previous Cholesky panel (see k_chol_panel)
    double* Kc[VGGP_MAX_D];       // factored in place -> Cholesky factor (lower)
    double* W[VGGP_MAX_D];        // C^-1
    double* Lt[VGGP_MAX_D];       // tril(L_d)
    double* Q[VGGP_MAX_D];
    double* dP[VGGP_MAX_D];
    double* dR[VGGP_MAX_D];
    double* X[VGGP_MAX_D];
    double* Y[VGGP_MAX_D];
    double* dK[VGGP_MAX_D];
    double* dLraw[VGGP_MAX_D];
    double* tmp[VGGP_MAX_D];
    double* gen[VGGP_MAX_D];      // B1 plans only: generators of P_d, [pd | ru | rl] each n (k_b1_gens)
    double* sc;                   // SC_COUNT scalars
    int* info;
    void* bandT;                  // per-cell tables in obs dtype: per dim [pe0 pe1 pe2 qe0 qe1 qe2 h rh], each n[d] long
    int leaf_cnt[VGGP_MAX_D];
    int leaf_lo[VGGP_MAX_D][MAX_LEAVES + 1];
};

// ---------------------------------------------------------------------------------------------------------
// K_d(theta) entry.  theta = [l_1..l_D, s2_1..s2_D, noise].
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double b1_A(int i, int j, int n, double dl) {
    if (i == j) return (2.0 / 3.0 * dl) + ((i == 0 || i == n - 1) ? -(1.0 / 3.0 * dl) : 0.0);
    if (i - j == 1 || j - i == 1) return 1.0 / 6.0 * dl;
    return 0.0;
}
__device__ __forceinline__ double b1_B(int i, int j, int n, double dl) {
    if (i == j) return (2.0 / dl) + ((i == 0 || i == n - 1) ? -(1.0 / dl) : 0.0);
    if (i - j == 1 || j - i == 1) return -1.0 / dl;
    return 0.0;
}
__device__ __forceinline__ double b1_BC(int i, int j, int n) { return (i == j && (i == 0 || i == n - 1)) ? 1.0 : 0.0; }

// (k * delta) rounded to float32 first, as the reference's int64-tensor * 0-dim float32 does
__device__ __forceinline__ double b0_kdelta(int k, float delta32) { return (double)((float)k * delta32); }

// r(k) and d r(k) / d l of the B0 Toeplitz first row (without the l^2 s2 factor)
__device__ __forceinline__ void b0_row(int k, float delta32, double l, double& r, double& dr) {
    if (k == 0) {
        const double dl = (double)delta32;
        const double e = exp(-dl / l);
        r = 2.0 * (e + dl / l - 1.0);
        dr = 2.0 * (e * dl / (l * l) - dl / (l * l));
    } else {
        const double a0 = b0_kdelta(k - 1, delta32), a1 = b0_kdelta(k + 1, delta32), a2 = b0_kdelta(k, delta32);
        const double e0 = exp(-a0 / l), e1 = exp(-a1 / l), e2 = exp(-a2 / l);
        r = e0 + e1 - 2.0 * e2;
        const double il2 = 1.0 / (l * l);
        dr = (e0 * a0 + e1 * a1 - 2.0 * e2 * a2) * il2;
    }
}

__device__ __forceinline__ double factor_entry(const GridDims& g, const double* theta, int d, int i, int j) {
    const double l = theta[d], s2 = theta[g.D + d];
    const int n = g.n[d];
    if (g.family == VGGP_B1_ASVGP) {
        const double dl = (double)g.delta32[d];
        const int dist = i > j ? i - j : j - i;
        if (dist > 1) return 0.0;
        return (b1_A(i, j, n, dl) * l + b1_B(i, j, n, dl) * (1.0 / l) + b1_BC(i, j, n)) * (1.0 / (2.0 * s2));
    } else if (g.family == VGGP_SVGP_GRID) {
        // kernel_d(Z).evaluate(), kronecker_structure.py:321-322: ScaleKernel(MaternKernel(nu = 1/2)) at the inducing points
        return s2 * exp(-fabs((double)g.knots[d][i] - (double)g.knots[d][j]) / l);
    } else if (g.family == VGGP_VFF_GRID) {
        // DiagLinearOperator(alpha).add_low_rank(beta), kronecker_structure.py:403-462: alpha_i = (b - a) / 2 c_i / S(w_i) with
        // 1 / S(w) = (1 / l + w^2 l) / (2 s2), c_0 = 2; beta = 1 / sqrt(s2) on the M + 1 cosine rows, 0 on the M sine rows
        const int Mf = (n - 1) / 2;
        double v = (i <= Mf && j <= Mf) ? 1.0 / s2 : 0.0;
        if (i == j) {
            const double a = (double)g.knots[d][0], b = (double)g.knots[d][n - 1];
            const int kf = i <= Mf ? i : i - Mf;
            const double w = 6.283185307179586476925286766559 * (double)kf / (b - a);
            v += 0.5 * (b - a) * (i == 0 ? 2.0 : 1.0) * (1.0 / l + w * w * l) / (2.0 * s2);
        }
        return v;
    } else {
        double r, dr;
        b0_row(i > j ? i - j : j - i, g.delta32[d], l, r, dr);
        return r * (l * l * s2);
    }
}

// d K_d[i][j] / d l and / d s2
__device__ __forceinline__ void factor_entry_grad(const GridDims& g, const double* theta, int d, int i, int j,
                                                  double& dKdl, double& dKds2) {
    const double l = theta[d], s2 = theta[g.D + d];
    const int n = g.n[d];
    if (g.family == VGGP_B1_ASVGP) {
        const double dl = (double)g.delta32[d];
        const int dist = i > j ? i - j : j - i;
        if (dist > 1) { dKdl = 0.0; dKds2 = 0.0; return; }
        const double A = b1_A(i, j, n, dl), B = b1_B(i, j, n, dl), BC = b1_BC(i, j, n);
        dKdl = (A - B / (l * l)) / (2.0 * s2);
        dKds2 = -(A * l + B / l + BC) / (2.0 * s2 * s2);
    } else if (g.family == VGGP_SVGP_GRID) {
        const double a = fabs((double)g.knots[d][i] - (double)g.knots[d][j]), e = exp(-a / l);
        dKdl = s2 * e * a / (l * l);
        dKds2 = e;
    } else if (g.family == VGGP_VFF_GRID) {
        const int Mf = (n - 1) / 2;
        dKdl = 0.0;
        dKds2 = (i <= Mf && j <= Mf) ? -1.0 / (s2 * s2) : 0.0;
        if (i == j) {
            const double a = (double)g.knots[d][0], b = (double)g.knots[d][n - 1];
            const int kf = i <= Mf ? i : i - Mf;
            const double w = 6.283185307179586476925286766559 * (double)kf / (b - a);
            const double c = 0.5 * (b - a) * (i == 0 ? 2.0 : 1.0);
            dKdl = c * (-1.0 / (l * l) + w * w) / (2.0 * s2);
            dKds2 -= c * (1.0 / l + w * w * l) / (2.0 * s2 * s2);
        }
    } else {
        double r, dr;
        b0_row(i > j ? i - j : j - i, g.delta32[d], l, r, dr);
        dKdl = s2 * (2.0 * l * r + l * l * dr);
        dKds2 = l * l * r;
    }
}

// grid (ceil(nmax^2 / 256), D)
__global__ void k_build_factors(const __grid_constant__ GridDims g, const double* __restrict__ theta,
                                const double* __restrict__ L) {
    const int d = blockIdx.y;
    const int n = g.n[d];
    const i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (blockIdx.x == 0 && d == 0 && threadIdx.x < SC_COUNT) g.sc[threadIdx.x] = 0.0;
    if (blockIdx.x == 0 && d == 0 && threadIdx.x == 0) *g.info = 0;
    if (e >= (i64)n * n) return;
    const int i = (int)(e / n), j = (int)(e % n);
    const double k = factor_entry(g, theta, d, i, j);
    g.Kraw[d][e] = k;
    g.Kc[d][e] = k;
    g.W[d][e] = 0.0;
    g.Lt[d][e] = (j <= i) ? L[g.Loff[d] + e] : 0.0;
}

// ---------------------------------------------------------------------------------------------------------
// Blocked right-looking Cholesky, one panel per launch: every CTA factors the NB x NB diagonal block in
// shared memory (redundantly -- it is tiny), CTA 0 keeps the result and accumulates the log-det, CTA c >= 1
// solves its NB rows of the panel against it.  The trailing update is a grouped GEMM launch.
// CTA 0 must not overwrite the diagonal block in place while the other CTAs of the launch may still have to read
// the unfactored block (nothing orders CTAs of one launch; sequential execution of the blocks, as under the test
// emulator, reads a half-factored block): unless it is the only CTA of its dimension it parks the factor in
// g.cdiag[d], and CTA 0 of the next panel launch moves it into place (nothing in between reads that block).
// grid (row chunks, D), 256 threads, dynamic smem (2 * NB * CHOL_PITCH + 2 * NB) doubles.
// ---------------------------------------------------------------------------------------------------------
constexpr int CHOL_PITCH = NB + 4;      // 4 lanes per row read s[r][q], s[r][q + 4], ...: pitch = 4 (mod 16) doubles keeps them on distinct banks
__global__ void __launch_bounds__(256) k_chol_panel(const __grid_constant__ GridDims g, int j0) {
    extern __shared__ double sm[];
    double (*s)[CHOL_PITCH] = reinterpret_cast<double (*)[CHOL_PITCH]>(sm);
    double (*a)[CHOL_PITCH] = reinterpret_cast<double (*)[CHOL_PITCH]>(sm + NB * CHOL_PITCH);
    double* dg = sm + 2 * NB * CHOL_PITCH;    // the diagonal of the factor: kept apart until the block is done (see below)
    double* idg = dg + NB;                    // and its reciprocals, for the panel rows
    const int d = blockIdx.y;
    const int n = g.n[d];
    if (j0 >= n) return;
    const int w = min(NB, n - j0);
    const int r0 = j0 + (int)blockIdx.x * NB;
    if (r0 >= n) return;
    double* __restrict__ A = g.Kc[d];
    const int tid = threadIdx.x, nt = blockDim.x;

    if (blockIdx.x == 0 && j0 > 0) {          // the previous panel's diagonal factor, parked by its CTA 0 (full NB x NB block)
        for (int e = tid; e < NB * NB; e += nt) {
            const int i = e / NB, j = e % NB;
            if (j <= i) A[(i64)(j0 - NB + i) * n + (j0 - NB + j)] = g.cdiag[d][e];
        }
    }
    for (int e = tid; e < w * w; e += nt) {
        const int i = e / w, j = e % w;
        s[i][j] = A[(i64)(j0 + i) * n + (j0 + j)];
    }
    __syncthreads();
    // Left-looking factorisation of the diagonal block, 4 lanes per row (256 threads = 64 rows): column c of row r is
    // s[r][c] - sum_{k<c} s[r][k] s[c][k], the lanes split k modulo 4 and meet by two shuffles.  Every row group also forms the
    // pivot sum_{k<c} s[c][k]^2 itself (same operations in the same order: bit-identical everywhere), so one barrier per
    // column is enough -- the right-looking version needed three and ran at 1.4 us per column.  The new diagonal entry goes
    // to dg[c], not to s[c][c]: the other row groups read s[c][c] in the same iteration.
    const int r = tid >> 2, q = tid & 3;
    for (int c = 0; c < w; ++c) {
        double part = 0.0, pp = 0.0;
        if (r >= c && r < w) {
            for (int k = q; k < c; k += 4) {
                const double sc = s[c][k];
                part = fma(s[r][k], sc, part);
                pp = fma(sc, sc, pp);
            }
        }
        part += __shfl_xor_sync(0xffffffffu, part, 1);
        pp += __shfl_xor_sync(0xffffffffu, pp, 1);
        part += __shfl_xor_sync(0xffffffffu, part, 2);
        pp += __shfl_xor_sync(0xffffffffu, pp, 2);
        if (r >= c && r < w && q == 0) {
            const double piv = s[c][c] - pp;
            // one reciprocal square root per row instead of a square root and a division (both software sequences in float64);
            // a Newton step makes it as accurate as 1 / sqrt computed separately
            double rs = rsqrt(piv);
            rs = fma(rs * 0.5, fma(-piv * rs, rs, 1.0), rs);
            if (r == c) {
                if (!(piv > 0.0)) atomicMax(g.info, d + 1);
                dg[c] = piv * rs;
                idg[c] = rs;
            } else {
                s[r][c] = (s[r][c] - part) * rs;
            }
        }
        __syncthreads();
    }
    if (tid < w) s[tid][tid] = dg[tid];
    __syncthreads();
    if (blockIdx.x == 0) {
        const bool alone = j0 + NB >= n;      // last panel of this dimension: no other CTA reads the block
        for (int e = tid; e < w * w; e += nt) {
            const int i = e / w, j = e % w;
            if (j <= i) {
                if (alone) A[(i64)(j0 + i) * n + (j0 + j)] = s[i][j];
                else g.cdiag[d][i * NB + j] = s[i][j];          // w == NB here
            }
        }
        if (tid == 0) {
            double ld = 0.0;
            for (int c = 0; c < w; ++c) ld += log(s[c][c]);
            g.sc[SC_LOGDETK + d] += 2.0 * ld;     // single writer per launch; launches are stream-ordered
        }
        return;
    }
    const int rows = min(NB, n - r0);
    for (int e = tid; e < rows * w; e += nt) {
        const int i = e / w, j = e % w;
        a[i][j] = A[(i64)(r0 + i) * n + (j0 + j)];
    }
    __syncthreads();
    // rows of the panel against the factored block: independent rows, 4 lanes each (all in one warp: __syncwarp orders them)
    for (int c = 0; c < w; ++c) {
        double part = 0.0;
        if (r < rows)
            for (int k = q; k < c; k += 4) part = fma(a[r][k], s[c][k], part);
        part += __shfl_xor_sync(0xffffffffu, part, 1);
        part += __shfl_xor_sync(0xffffffffu, part, 2);
        if (r < rows && q == 0) a[r][c] = (a[r][c] - part) * idg[c];
        __syncwarp();
    }
    __syncthreads();
    for (int e = tid; e < rows * w; e += nt) {
        const int i = e / w, j = e % w;
        A[(i64)(r0 + i) * n + (j0 + j)] = a[i][j];
    }
}

// Inverse of the diagonal (leaf) blocks of the lower-triangular factor: W[lo:hi, lo:hi] = C[lo:hi, lo:hi]^-1.
// grid (max leaves, D), NB threads, dynamic smem 2 * NB * (NB+1) doubles.
__global__ void __launch_bounds__(NB) k_triinv_leaf(const __grid_constant__ GridDims g) {
    extern __shared__ double sm[];
    double (*c)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(sm);
    double (*x)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(sm + NB * (NB + 1));
    const int d = blockIdx.y;
    if ((int)blockIdx.x >= g.leaf_cnt[d]) return;
    const int n = g.n[d];
    const int lo = g.leaf_lo[d][blockIdx.x], hi = g.leaf_lo[d][blockIdx.x + 1];
    const int w = hi - lo;
    const double* __restrict__ C = g.Kc[d];
    double* __restrict__ W = g.W[d];
    const int tid = threadIdx.x;
    for (int e = tid; e < w * w; e += NB) {
        const int i = e / w, j = e % w;
        c[i][j] = (j <= i) ? C[(i64)(lo + i) * n + (lo + j)] : 0.0;
    }
    __syncthreads();
    if (tid < w) {
        const int j = tid;
        x[j][j] = 1.0 / c[j][j];
        for (int i = j + 1; i < w; ++i) {
            double v = 0.0;
            for (int k = j; k < i; ++k) v -= c[i][k] * x[k][j];
            x[i][j] = v / c[i][i];
        }
        for (int i = j; i < w; ++i) W[(i64)(lo + i) * n + (lo + j)] = x[i][j];
    }
}

// ---------------------------------------------------------------------------------------------------------
// Forward reductions, one warp per row i of dimension d: per-cell tables of P_d and Q_d (observation dtype,
// monomial basis), the float64 band of Q_d, tr(P_d S_d) = <R_d, tril L_d>, log det S_d = 2 sum log |L_ii|.
// The band of Q_d = R_d R_d^T is formed from row dot products.
// grid (ceil(nmax / 8), D), 256 threads.
// ---------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_fwd_reduce(const __grid_constant__ GridDims g) {
    const int d = blockIdx.y;
    const int n = g.n[d];
    const int lane = threadIdx.x & 31;
    const int i = (int)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= n) return;
    const double* __restrict__ P = g.P[d];
    const double* __restrict__ R = g.R[d];
    const double* __restrict__ Lt = g.Lt[d];
    const bool last = (i + 1 >= n);
    double qd = 0.0, qo = 0.0, tr = 0.0;
    const double* Ri = R + (i64)i * n;
    const double* Rn = R + (i64)(last ? i : i + 1) * n;
    const double* Li = Lt + (i64)i * n;
    for (int k = lane; k < n; k += 32) {
        const double r = Ri[k];
        qd = fma(r, r, qd);
        qo = fma(r, Rn[k], qo);
        tr = fma(r, Li[k], tr);
    }
    qd = warp_sum(qd);
    qo = warp_sum(qo);
    tr = warp_sum(tr);
    if (lane == 0) {
        if (last) qo = 0.0;
        g.Qb[d][i] = qd;
        g.Qb[d][n + i] = qo;
        // per-cell tables, monomial basis in the hat weight a (w_lo = 1 - a):
        //   p(a) = A (1-a)^2 + 2 B (1-a) a + C a^2 = pe0 + pe1 a + pe2 a^2, A = P[c][c], B = P[c][c+1], C = P[c+1][c+1]
        T* tab = reinterpret_cast<T*>(g.bandT) + g.tab_off[d];       // [pe0 | pe1 | pe2 | qe0 | qe1 | qe2 | h | rh]
        const double A = P[(i64)i * n + i];
        const double B2 = last ? 0.0 : 2.0 * P[(i64)i * n + i + 1];
        const double C = last ? 0.0 : P[(i64)(i + 1) * n + i + 1];
        tab[i] = (T)A; tab[n + i] = (T)(B2 - 2.0 * A); tab[2 * n + i] = (T)(A - B2 + C);
        atomicAdd(g.sc + SC_TR + d, tr);
        atomicAdd(g.sc + SC_LOGDETS + d, 2.0 * log(fabs(Li[i])));
    }
}

// Second half of the per-cell tables: needs Q[c+1][c+1] of the next row, so it runs after k_fwd_reduce.
// grid (ceil(nmax / 256), D)
template <typename T>
__global__ void __launch_bounds__(256) k_fwd_qtable(const __grid_constant__ GridDims g) {
    const int d = blockIdx.y;
    const int n = g.n[d];
    const int i = (int)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const bool last = (i + 1 >= n);
    T* tab = reinterpret_cast<T*>(g.bandT) + g.tab_off[d];
    const double Aq = g.Qb[d][i], B2q = last ? 0.0 : 2.0 * g.Qb[d][n + i], Cq = last ? 0.0 : g.Qb[d][i + 1];
    tab[3 * n + i] = (T)Aq; tab[4 * n + i] = (T)(B2q - 2.0 * Aq); tab[5 * n + i] = (T)(Aq - B2q + Cq);
}

// alpha (float64) -> observation dtype, and <m, alpha>.
template <typename T>
__global__ void __launch_bounds__(256) k_cast_alpha(const double* __restrict__ alpha, const double* __restrict__ m,
                                                    T* __restrict__ alphaT, i64 M, double* __restrict__ sc) {
    __shared__ double red[32];
    double acc = 0.0;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (i64)gridDim.x * blockDim.x) {
        const double a = alpha[i];
        alphaT[i] = (T)a;
        acc += a * m[i];
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) atomicAdd(sc + SC_MALPHA, acc);
}

// ---------------------------------------------------------------------------------------------------------
// Reverse pass pieces
// ---------------------------------------------------------------------------------------------------------
struct GbufView {
    const void* obs;       // n_obs_elems values of the observation dtype: [g_alpha (M) | band blocks]
    const double* scal;    // float64 scalars
};

// g = (ell_scale / noise) * g_alpha_raw, ghat = g - m/2
template <typename T>
__global__ void __launch_bounds__(256) k_bwd_prep(const T* __restrict__ ga, const double* __restrict__ m,
                                                  const double* __restrict__ theta, int D, double ell_scale,
                                                  double* __restrict__ gout, double* __restrict__ ghat, i64 M) {
    const double c = ell_scale / theta[2 * D];
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (i64)gridDim.x * blockDim.x) {
        const double v = c * (double)ga[i];
        gout[i] = v;
        ghat[i] = v - 0.5 * m[i];
    }
}

__device__ __forceinline__ double tr_others(const GridDims& g, int d) {
    double c = 1.0;
    for (int e = 0; e < g.D; ++e)
        if (e != d) c *= g.sc[SC_TR + e];
    return c;
}

// Dense-feature (B0) family: the per-observation kernel returns FULL factor-gradient sums bP_d, bQ_d.
//   dP_d += cP bP_d ;  X_d = cQ (bQ_d + bQ_d^T) = 2 cQ sym(bQ_d)   (then dR_d = X_d R_d by a GEMM)
// grid (ceil(nmax^2/256), D)
template <typename T>
__global__ void __launch_bounds__(256) k_bwd_dense_prep(const __grid_constant__ GridDims g, const T* __restrict__ gfac,
                                                        const double* __restrict__ theta, double ell_scale) {
    const int d = blockIdx.y;
    const int n = g.n[d];
    const i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (i64)n * n) return;
    const int i = (int)(e / n), j = (int)(e % n);
    const double noise = theta[2 * g.D];
    const double cP = ell_scale / (2.0 * noise), cQ = -ell_scale / (2.0 * noise);
    const T* __restrict__ bP = gfac + g.gfac_off[d];
    const T* __restrict__ bQ = bP + (i64)n * n;
    g.dP[d][e] += cP * (double)bP[e];
    g.X[d][e] = cQ * ((double)bQ[e] + (double)bQ[(i64)j * n + i]);
}

// X = (dP + dP^T) / 2.   grid (ceil(nmax^2/256), D)
__global__ void __launch_bounds__(256) k_sym(const __grid_constant__ GridDims g) {
    const int d = blockIdx.y;
    const int n = g.n[d];
    const i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (i64)n * n) return;
    const int i = (int)(e / n), j = (int)(e % n);
    g.X[d][e] = 0.5 * (g.dP[d][e] + g.dP[d][(i64)j * n + i]);
}

// dL_out = tril(dLraw - c_d R_d + (M/M_d) diag(1/L_ii)).   grid (ceil(nmax^2/256), D)
__global__ void __launch_bounds__(256) k_bwd_dL(const __grid_constant__ GridDims g, double* __restrict__ dL) {
    const int d = blockIdx.y;
    const int n = g.n[d];
    const i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (i64)n * n) return;
    const int i = (int)(e / n), j = (int)(e % n);
    double v = 0.0;
    if (j <= i) {
        v = g.dLraw[d][e] - tr_others(g, d) * g.R[d][e];
        if (i == j) v += ((double)g.M / (double)n) / g.Lt[d][e];
    }
    dL[g.Loff[d] + e] = v;
}

// dm = (kron P) g - alpha
__global__ void __launch_bounds__(256) k_bwd_dm(const double* __restrict__ pg, const double* __restrict__ alpha,
                                                double* __restrict__ dm, i64 M) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (i64)gridDim.x * blockDim.x)
        dm[i] = pg[i] - alpha[i];
}

// d theta and the ELBO scalars.
//   dK_d(total) = -Y_d P_d + (c_d / 2) Q_d - (M / (2 M_d)) P_d,  Y_d = P_d sym(dP_d),  c_d = prod_{e != d} tr(P_e S_e)
//   dl_d = <dK, dK/dl>, ds2_d = <dK, dK/ds2> + dkff * kff / s2_d        (accumulated atomically into dtheta)
// dK_d = -Y_d P_d comes from a GEMM.
// grid (chunks, D), 256 threads; dtheta must be zero on entry.  Block (0, 0) also writes dnoise and out[0..3].
__global__ void __launch_bounds__(256) k_bwd_theta(const __grid_constant__ GridDims g, const double* __restrict__ theta,
                                                   const double* __restrict__ gscal, double ell_scale,
                                                   double* __restrict__ out, double* __restrict__ dtheta) {
    __shared__ double red[32];
    const int d = blockIdx.y;
    const int n = g.n[d];
    const int D = g.D;
    const double* __restrict__ P = g.P[d];
    const double half_ratio = 0.5 * (double)g.M / (double)n;
    const double half_c = 0.5 * tr_others(g, d);
    const double* __restrict__ dK = g.dK[d];
    const double* __restrict__ Q = g.Q[d];
    double sl = 0.0, ss = 0.0;
    for (i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x; e < (i64)n * n; e += (i64)gridDim.x * blockDim.x) {
        const int i = (int)(e / n), j = (int)(e % n);
        double a, b;
        factor_entry_grad(g, theta, d, i, j, a, b);
        const double v = dK[e] + half_c * Q[e] - half_ratio * P[e];
        sl += v * a;
        ss += v * b;
    }
    sl = block_sum(sl, red);
    ss = block_sum(ss, red);
    if (threadIdx.x == 0) {
        atomicAdd(dtheta + d, sl);
        atomicAdd(dtheta + D + d, ss);
        if (blockIdx.x == 0) {
            const double noise = theta[2 * D];
            double kff = 1.0;
            for (int e = 0; e < D; ++e) kff *= theta[D + e];
            const double E = gscal[0], nobs = gscal[1];
            const double dkff = -ell_scale * nobs / (2.0 * noise);
            atomicAdd(dtheta + D + d, dkff * kff / theta[D + d]);
            // the features themselves depend on (l_d, s2_d): sums accumulated by the per-observation kernel
            atomicAdd(dtheta + d, (ell_scale / noise) * gscal[3 + d]);
            if (g.family != VGGP_VFF_GRID)      // Fourier features do not scale with s2_d (phi = s2 * ... in the other families)
                atomicAdd(dtheta + D + d, (ell_scale / noise) * gscal[5 + d] / theta[D + d]);
            if (d == 0) {
                const double tot = E + nobs * kff;
                const double ell = -0.5 * nobs * log(2.0 * 3.14159265358979323846 * noise) - tot / (2.0 * noise);
                atomicAdd(dtheta + 2 * D, ell_scale * (-nobs / (2.0 * noise) + tot / (2.0 * noise * noise)));
                double trp = 1.0, lds = 0.0;
                for (int e = 0; e < D; ++e) {
                    trp *= g.sc[SC_TR + e];
                    lds += ((double)g.M / (double)g.n[e]) * (g.sc[SC_LOGDETK + e] - g.sc[SC_LOGDETS + e]);
                }
                const double kl = 0.5 * (trp + g.sc[SC_MALPHA] - (double)g.M + lds);
                out[0] = ell_scale * ell - kl;
                out[1] = ell_scale * ell;
                out[2] = kl;
                out[3] = nobs;
            }
        }
    }
}

}  // namespace vggp
