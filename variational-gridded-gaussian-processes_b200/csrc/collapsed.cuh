// Collapsed ELBO of the B1 (ASVGP) and VGGP_SVGP_MARKOV families at any grid size (DESIGN.md section 4, K1l).
//
// With A = F + G / noise the system of the optimal mean (meanopt.cuh: F = Kuu for B1, F = Kuu^-1 for Markov; both are
// kron_d F_d with tridiagonal F_d), the reference's collapsed bound is, by the matrix determinant lemma,
//     ELBO = -1/2 [ N log 2 pi + N log noise + log det A - log det F + (y^T y - b^T x*) / noise ]
//            - (N prod_d s2_d - tr(F^-1 G)) / (2 noise)
// (B1: log det F = log det Kuu, tr(Kuu^-1 G); Markov: log det F = -log det Kuu, tr(Kuu G)).  x* is the solver's iterate of
// the mean system.  Everything but log det A is exact; the terms kernels below compute it in one pass over the binned data
// and the grid.  log det A is estimated by preconditioned stochastic Lanczos quadrature: with the preconditioner P = C C^T,
//     log det A = log det P + tr log B,   B = C^-1 A C^-T,
//     Kronecker: C = kron_d L_d D_d^(1/2) of the Thomas factors of F_d + g I (meanopt.cuh), log det P = sum_d (M / M_d) sum_i log d'_i
//     Jacobi:    C = diag(A)^(1/2),                                                           log det P = sum_u log A_uu
// and tr log B ~ mean_j eps_j^T log(B) eps_j from the Lanczos tridiagonal T_j of each probe (Gauss quadrature on the host).
// The k probes are one [k][M] block; every reduction is per-CTA partials summed in a fixed order (no floating-point
// atomics), so one assembled system and one seed give the same bits from call to call.
#pragma once
#include "meanopt.cuh"
#include "minibatch.cuh"

namespace vggp {

// Rademacher sign of node u of probe j: the 32-bit mixing hash of minibatch.cuh keyed by (seed, probe)
__host__ __device__ __forceinline__ uint32_t ct_probe_key(uint64_t seed, int probe) {
    uint32_t h = mb_mix32((uint32_t)seed);
    h = mb_mix32(h ^ (uint32_t)(seed >> 32));
    return mb_mix32(h ^ (uint32_t)(probe + 1) * 0x9e3779b9u);
}
__host__ __device__ __forceinline__ double ct_sign(uint32_t key, i64 u) {
    return (mb_mix32(key ^ (uint32_t)u) >> 31) ? -1.0 : 1.0;
}

}  // namespace vggp

#if (defined(__CUDACC__) || defined(VGGP_EMUL)) && !defined(VGGP_HOST_EMUL)
namespace vggp {

constexpr int CT_THREADS = 256;

// Lanczos state of k probes.  Vectors [k][M]; coefficients [probe][step]; `done` is set by the host once a probe's
// quadrature has converged, or by k_ct_beta when the Krylov space is exhausted (beta ~ 0) or the step limit is reached.
struct CtLanczos {
    i64 M;
    int k, max_steps;
    double *alpha, *beta;        // [k][max_steps]
    int* nsteps;                 // [k] steps taken
    int* done;                   // [k]
    double* part;                // [2 k][nb] per-CTA partial sums (rows j: y . v1, rows k + j: ||y||^2)
    int nb;                      // CTAs per probe of k_ct_dot / k_ct_update
};

// v1 = eps_j / ||eps_j||, v0 = 0.  kind 0: Rademacher (||eps|| = sqrt M); 1: e_{first + j}
__global__ void __launch_bounds__(CT_THREADS) k_ct_probe_init(i64 M, int kind, uint64_t seed_or_first, double* __restrict__ v0,
                                                              double* __restrict__ v1) {
    const int j = blockIdx.y;
    const uint32_t key = ct_probe_key(seed_or_first, j);
    const double scale = 1.0 / sqrt((double)M);
    const i64 unit = (i64)seed_or_first + j;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < M; u += (i64)gridDim.x * blockDim.x) {
        v0[(i64)j * M + u] = 0.0;
        v1[(i64)j * M + u] = kind == 0 ? scale * ct_sign(key, u) : (u == unit ? 1.0 : 0.0);
    }
}

// d'^-1/2 of every dimension's Thomas factors (fac + fac_off[d] + n_d: 1 / d'), at rs + off[d] / 3
template <int D>
__global__ void __launch_bounds__(CT_THREADS) k_ct_rsqrt_pivots(const __grid_constant__ MoSys<D> s, const double* __restrict__ fac,
                                                                const __grid_constant__ MoFacOff<D> fo, double* __restrict__ rs) {
    const int d = blockIdx.y, n = s.n[d];
    const int i = (int)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rs[fo.off[d] / 3 + i] = sqrt(fac[fo.off[d] + n + i]);
}

// One mode of C^-1 (FWD) or C^-T (BWD) on every fibre of the [k][M] probe block, in place or from `in` to `out`:
//   FWD:  y_i = x_i - l_i y_{i-1},  out_i = y_i d'_i^-1/2                    (D^-1/2 L^-1)
//   BWD:  z_i = x_i d'_i^-1/2 - l_{i+1} z_{i+1},  out_i = z_i                 (L^-T D^-1/2)
// The segmented scheme of k_mo_kron_sweep (meanopt.cuh) with one recurrence instead of two: each fibre is cut into S segments,
// one thread per (fibre, segment); the affine map of a segment is composed from a zero start (one read), the maps of the
// earlier (FWD) or later (BWD) segments of the fibre are chained in shared memory into the segment's start value, and the
// exact recurrence runs from it (one read, one write).  STAGED (the contiguous mode): the block's rows are copied into shared
// memory with coalesced loads, swept there and written back the same way; the launch shape is mo_sweep_cfg's with the k M / n
// fibres of the block.  Fibres of a finished probe are left as they are.
template <bool FWD, bool STAGED>
__global__ void __launch_bounds__(1024) k_ct_kron_half(const __grid_constant__ MoSweep w, i64 M, const double* __restrict__ rs,
                                                       const double* in, double* out, const int* __restrict__ done) {
    __shared__ double sa[1024], sb[1024];
    extern __shared__ double sm[];
    const int tid = threadIdx.x, S = w.S, FB = (int)blockDim.x / S, n = w.n;
    const int seg = STAGED ? tid % S : tid / FB, fl = STAGED ? tid / S : tid % FB;
    const i64 f0 = (i64)blockIdx.x * FB, f = f0 + fl;
    const int lo = min(n, seg * w.Ls), hi = min(n, lo + w.Ls);
    const double* __restrict__ l = w.fac;
    const double* src;
    double* dst;
    i64 step, base;
    const i64 nrows = min((i64)FB, w.F - f0);
    if (STAGED) {
        for (i64 j = tid; j < nrows * n; j += blockDim.x) {
            const int row = (int)(j / n), i = (int)(j - (i64)row * n);
            sm[(i64)row * S * w.P + (i / w.Ls) * w.P + i % w.Ls] = in[f0 * n + j];
        }
        __syncthreads();
        dst = sm + (i64)fl * S * w.P + (i64)(seg * w.P) - lo;
        src = dst;
        step = 1;
        base = f * n;
    } else {
        const i64 outer = f / w.inner, j = f - outer * w.inner;
        base = outer * n * w.inner + j;
        src = in + base;
        dst = out + base;
        step = w.inner;
    }
    const bool act = f < w.F && !done[base / M];
    auto idx = [&](int s2) { return STAGED ? fl * S + s2 : s2 * FB + fl; };
    double A = 1.0, B = 0.0, c = 0.0;
    if (FWD) {
        if (S > 1) {            // y_{hi-1} = A y_{lo-1} + B
            if (act)
                for (int i = lo; i < hi; ++i) { B = fma(-l[i], B, src[i * step]); A *= -l[i]; }
            sa[tid] = A; sb[tid] = B;
            __syncthreads();
            for (int s2 = 0; s2 < seg; ++s2) c = fma(sa[idx(s2)], c, sb[idx(s2)]);
        }
        if (act)
            for (int i = lo; i < hi; ++i) {
                c = fma(-l[i], c, src[i * step]);
                dst[i * step] = c * rs[i];
            }
    } else {
        if (S > 1) {            // z_lo = A z_hi + B
            if (act)
                for (int i = hi - 1; i >= lo; --i) {
                    const double li = i + 1 < n ? l[i + 1] : 0.0;
                    B = fma(-li, B, src[i * step] * rs[i]);
                    A *= -li;
                }
            sa[tid] = A; sb[tid] = B;
            __syncthreads();
            for (int s2 = S - 1; s2 > seg; --s2) c = fma(sa[idx(s2)], c, sb[idx(s2)]);
        }
        if (act)
            for (int i = hi - 1; i >= lo; --i) {
                const double li = i + 1 < n ? l[i + 1] : 0.0;
                c = fma(-li, c, src[i * step] * rs[i]);
                dst[i * step] = c;
            }
    }
    if (STAGED) {
        __syncthreads();
        for (i64 j = tid; j < nrows * n; j += blockDim.x) {
            const int row = (int)(j / n), i = (int)(j - (i64)row * n);
            out[f0 * n + j] = sm[(i64)row * S * w.P + (i / w.Ls) * w.P + i % w.Ls];
        }
    }
}

// out_j = A in_j for every live probe (JAC: out_j = S A S in_j, S = diag(A)^-1/2 in `sdiag`).  The 3^D coefficients of a row
// (the stencil of mo_row) are formed once and applied to all k vectors.
template <int D, bool JAC>
__global__ void __launch_bounds__(CT_THREADS) k_ct_stencil(const __grid_constant__ MoSys<D> s, int k, const double* __restrict__ in,
                                                           double* __restrict__ out, const double* __restrict__ sdiag,
                                                           const int* __restrict__ done) {
    constexpr int P3 = Pow3<D>::v, KC = (P3 - 1) / 2;
    const double inv_noise = 1.0 / s.theta[2 * D];
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < s.M; u += (i64)gridDim.x * blockDim.x) {
        int idx[D];
        {
            i64 rem = u;
#pragma unroll
            for (int d = 0; d < D; ++d) { idx[d] = (int)(rem / s.stride[d]); rem -= (i64)idx[d] * s.stride[d]; }
        }
        double c[D][3];
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const int i = idx[d];
            c[d][1] = s.bd[d][i];
            c[d][0] = i > 0 ? s.bo[d][i - 1] : 0.0;
            c[d][2] = i + 1 < s.n[d] ? s.bo[d][i] : 0.0;
        }
        double cp[P3];
        i64 off[P3];
#pragma unroll
        for (int q = 0; q < P3; ++q) {
            int kk = q;
            i64 o = 0;
            bool ok = true;
            double v = 1.0;
#pragma unroll
            for (int d = D - 1; d >= 0; --d) {
                const int od = kk % 3;
                kk /= 3;
                const int jn = idx[d] + od - 1;
                ok = ok && jn >= 0 && jn < s.n[d];
                o += (i64)(od - 1) * s.stride[d];
                v *= c[d][od];
            }
            if (ok) {
                v += inv_noise * (q >= KC ? s.G[(i64)(q - KC) * s.M + u] : s.G[(i64)(P3 - 1 - q - KC) * s.M + u + o]);
                if (JAC) v *= sdiag[u + o];
            } else {
                v = 0.0;
                o = 0;
            }
            cp[q] = v;
            off[q] = o;
        }
        const double su = JAC ? sdiag[u] : 1.0;
        for (int j = 0; j < k; ++j) {
            if (done[j]) continue;
            const double* x = in + (i64)j * s.M + u;
            double acc = 0.0;
#pragma unroll
            for (int q = 0; q < P3; ++q) acc = fma(cp[q], x[off[q]], acc);
            out[(i64)j * s.M + u] = su * acc;
        }
    }
}

// diag(A)^-1/2 for the Jacobi operator, and log A_uu into per-CTA partials (logdet P)
template <int D>
__global__ void __launch_bounds__(CT_THREADS) k_ct_jacobi(const __grid_constant__ MoSys<D> s, double* __restrict__ sdiag,
                                                          double* __restrict__ part) {
    __shared__ double red[32];
    const double inv_noise = 1.0 / s.theta[2 * D];
    double acc = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < s.M; u += (i64)gridDim.x * blockDim.x) {
        double dg = 1.0;
#pragma unroll
        for (int d = 0; d < D; ++d) {
            i64 rem = u / s.stride[d];
            dg *= s.bd[d][rem % s.n[d]];
        }
        dg += inv_noise * s.G[u];
        sdiag[u] = 1.0 / sqrt(dg);
        acc += log(dg);
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) part[blockIdx.x] = acc;
}

// fixed-order sum of n partials by one block; the result in every thread
__device__ __forceinline__ double ct_sum_partials(const double* __restrict__ p, int n, double* red, double* bc) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) acc += p[i];
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) *bc = acc;
    __syncthreads();
    return *bc;
}

// trace of G (slot 0) in a fixed order, for the shift g of the Kronecker factors: per-CTA partials, then k->gsum
__global__ void __launch_bounds__(CT_THREADS) k_ct_gtrace(i64 M, const double* __restrict__ G, double* __restrict__ part) {
    __shared__ double red[32];
    double acc = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < M; u += (i64)gridDim.x * blockDim.x) acc += G[u];
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) part[blockIdx.x] = acc;
}
__global__ void __launch_bounds__(CT_THREADS) k_ct_gtrace_final(const double* __restrict__ part, int nb, MoKron* k) {
    __shared__ double red[32], bc;
    const double v = ct_sum_partials(part, nb, red, &bc);
    if (threadIdx.x == 0) k->gsum = v;
}

// partial sums of y_j . v1_j into row j of the partials
__global__ void __launch_bounds__(CT_THREADS) k_ct_dot(const __grid_constant__ CtLanczos z, const double* __restrict__ y,
                                                       const double* __restrict__ v1) {
    __shared__ double red[32];
    const int j = blockIdx.y;
    if (z.done[j]) return;
    double acc = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < z.M; u += (i64)gridDim.x * blockDim.x)
        acc = fma(y[(i64)j * z.M + u], v1[(i64)j * z.M + u], acc);
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) z.part[(i64)j * z.nb + blockIdx.x] = acc;
}

// alpha_j = the fixed-order sum of row j of the partials; one block per probe
__global__ void __launch_bounds__(CT_THREADS) k_ct_alpha(const __grid_constant__ CtLanczos z, int step) {
    __shared__ double red[32], bc;
    const int j = blockIdx.x;
    if (z.done[j]) return;
    const double a = ct_sum_partials(z.part + (i64)j * z.nb, z.nb, red, &bc);
    if (threadIdx.x == 0) {
        z.alpha[(i64)j * z.max_steps + step] = a;
        z.nsteps[j] = step + 1;
    }
}

// y -= alpha_j v1 + beta_{j-1} v0; partial sums of ||y||^2 into row k + j
__global__ void __launch_bounds__(CT_THREADS) k_ct_update(const __grid_constant__ CtLanczos z, int step, double* __restrict__ y,
                                                          const double* __restrict__ v1, const double* __restrict__ v0) {
    __shared__ double red[32];
    const int j = blockIdx.y;
    if (z.done[j]) return;
    const double a = z.alpha[(i64)j * z.max_steps + step];
    const double b = step > 0 ? z.beta[(i64)j * z.max_steps + step - 1] : 0.0;
    double acc = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < z.M; u += (i64)gridDim.x * blockDim.x) {
        const i64 e = (i64)j * z.M + u;
        const double v = y[e] - a * v1[e] - b * v0[e];
        y[e] = v;
        acc = fma(v, v, acc);
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) z.part[(i64)(z.k + j) * z.nb + blockIdx.x] = acc;
}

// beta_j = ||y|| (fixed-order sum of row k + j); one block per probe.  A beta below 1e-13 |alpha_j| or the M-th step (the
// Krylov space is exhausted: the quadrature is exact) ends the probe with done = 2, the step limit with done = 3.
__global__ void __launch_bounds__(CT_THREADS) k_ct_beta(const __grid_constant__ CtLanczos z, int step) {
    __shared__ double red[32], bc;
    const int j = blockIdx.x;
    if (z.done[j]) return;
    const double bb = sqrt(ct_sum_partials(z.part + (i64)(z.k + j) * z.nb, z.nb, red, &bc));
    if (threadIdx.x == 0) {
        const double a = z.alpha[(i64)j * z.max_steps + step];
        z.beta[(i64)j * z.max_steps + step] = bb;
        const int end = (!(bb > 1e-13 * fabs(a)) || (i64)(step + 1) >= z.M) ? 2 : (step + 1 >= z.max_steps ? 3 : 0);
        if (end) z.done[j] = end;
    }
}

// y /= beta_j: the next v1
__global__ void __launch_bounds__(CT_THREADS) k_ct_next(const __grid_constant__ CtLanczos z, int step, double* __restrict__ y) {
    const int j = blockIdx.y;
    if (z.done[j]) return;
    const double r = 1.0 / z.beta[(i64)j * z.max_steps + step];
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < z.M; u += (i64)gridDim.x * blockDim.x) y[(i64)j * z.M + u] *= r;
}

// ---- exact terms ------------------------------------------------------------------------------------------------
// Band of F_d^-1 (diag | off, n each) and log det F_d for every dimension, one thread per dimension: with the pivots
// d_i of the top-down and e_i of the bottom-up elimination of the SPD tridiagonal F_d,
//     (F^-1)_ii = 1 / (d_i + e_i - F_ii),   (F^-1)_{i,i+1} = -F_{i,i+1} / (d_i e_{i+1} - F_{i,i+1}^2),   log det F = sum log d_i.
// `ib` holds 4 n values per dimension at offset 4 sum_{e < d} n_e: [diag | off | d | e].
template <int D>
__global__ void __launch_bounds__(32) k_ct_inv_bands(const __grid_constant__ MoSys<D> s, double* __restrict__ ib,
                                                     double* __restrict__ ldf) {
    const int d = threadIdx.x;
    if (d >= D) return;
    int o = 0;
    for (int e = 0; e < d; ++e) o += 4 * s.n[e];
    const int n = s.n[d];
    const double* a = s.bd[d];
    const double* b = s.bo[d];
    double* dg = ib + o;
    double* of = dg + n;
    double* dp = of + n;
    double* ep = dp + n;
    double ld = 0.0;
    dp[0] = a[0];
    ld += log(dp[0]);
    for (int i = 1; i < n; ++i) { dp[i] = a[i] - b[i - 1] * b[i - 1] / dp[i - 1]; ld += log(dp[i]); }
    ep[n - 1] = a[n - 1];
    for (int i = n - 2; i >= 0; --i) ep[i] = a[i] - b[i] * b[i] / ep[i + 1];
    for (int i = 0; i < n; ++i) {
        dg[i] = 1.0 / (dp[i] + ep[i] - a[i]);
        of[i] = i + 1 < n ? -b[i] / (dp[i] * ep[i + 1] - b[i] * b[i]) : 0.0;
    }
    ldf[d] = ld;
}

struct CtTermArgs {
    const unsigned char* data;   // data section of the binned buffer (obs dtype), `elems` values
    i64 elems;
    const double *b, *x;         // right-hand side b = sum w y and the solver's iterate
    const double* ib;            // k_ct_inv_bands
    double* part;                // [3][gridDim.x]
};

// per-CTA partials of { sum y^2 over the streamed data (padding holds y = 0), b . x, tr(F^-1 G) }
template <typename T, int D>
__global__ void __launch_bounds__(CT_THREADS) k_ct_terms(const __grid_constant__ MoSys<D> s, const __grid_constant__ CtTermArgs t) {
    constexpr int P3 = Pow3<D>::v, KC = (P3 - 1) / 2, GRP = (D + 1) * 128;
    __shared__ double red[32];
    const i64 tid = (i64)blockIdx.x * blockDim.x + threadIdx.x, nth = (i64)gridDim.x * blockDim.x;
    const T* data = reinterpret_cast<const T*>(t.data);
    double yy = 0.0, bx = 0.0, tr = 0.0;
    for (i64 e = tid; e < t.elems; e += nth)
        if (e % GRP >= D * 128) { const double y = (double)data[e]; yy = fma(y, y, yy); }
    int ioff[D];
    {
        int o = 0;
#pragma unroll
        for (int d = 0; d < D; ++d) { ioff[d] = o; o += 4 * s.n[d]; }
    }
    for (i64 u = tid; u < s.M; u += nth) {
        bx = fma(t.b[u], t.x[u], bx);
        int idx[D];
        i64 rem = u;
#pragma unroll
        for (int d = 0; d < D; ++d) { idx[d] = (int)(rem / s.stride[d]); rem -= (i64)idx[d] * s.stride[d]; }
#pragma unroll
        for (int q = KC; q < P3; ++q) {
            int kk = q;
            bool ok = true;
            double f = 1.0;
#pragma unroll
            for (int d = D - 1; d >= 0; --d) {
                const int od = kk % 3 - 1;
                kk /= 3;
                const int i = idx[d], jn = i + od;
                ok = ok && jn >= 0 && jn < s.n[d];
                if (ok) {
                    const double* dg = t.ib + ioff[d];
                    f *= od == 0 ? dg[i] : dg[s.n[d] + (od > 0 ? i : jn)];
                }
            }
            if (ok) tr = fma(q == KC ? 1.0 : 2.0, f * s.G[(i64)(q - KC) * s.M + u], tr);
        }
    }
    yy = block_sum(yy, red);
    bx = block_sum(bx, red);
    tr = block_sum(tr, red);
    if (threadIdx.x == 0) {
        t.part[blockIdx.x] = yy;
        t.part[gridDim.x + blockIdx.x] = bx;
        t.part[2 * gridDim.x + blockIdx.x] = tr;
    }
}

// out = { N, sum y^2 (+ the stored sum outside the mesh), b . x, tr(F^-1 G), log det Kuu }, one block, fixed order
template <int D>
__global__ void __launch_bounds__(CT_THREADS) k_ct_terms_final(const __grid_constant__ MoSys<D> s, const double* __restrict__ part,
                                                               int nb, const double* __restrict__ ldf, double n_obs,
                                                               const double* __restrict__ outside_yy, int markov,
                                                               double* __restrict__ out) {
    __shared__ double red[32], bc;
    double v[3];
    for (int r = 0; r < 3; ++r) v[r] = ct_sum_partials(part + (i64)r * nb, nb, red, &bc);
    if (threadIdx.x == 0) {
        double ld = 0.0;
        for (int d = 0; d < D; ++d) ld += ((double)s.M / (double)s.n[d]) * ldf[d];
        out[0] = n_obs;
        out[1] = v[0] + (outside_yy ? *outside_yy : 0.0);
        out[2] = v[1];
        out[3] = v[2];
        out[4] = markov ? -ld : ld;
    }
}

}  // namespace vggp
#endif
