// Optimal variational mean of the B1 (ASVGP) and VGGP_SVGP_MARKOV families (DESIGN.md section 4, K1m).
//
// The m-dependent part of the ELBO, -(1 / 2 noise) ||y - mu(m)||^2 - (1 / 2) m^T Kuu^-1 m, does not depend on S.  In both
// families an observation has non-zero weights w at the 2^D corners of its cell only, so its maximiser solves a symmetric
// positive definite 3^D-point stencil system on the node grid:
//     B1:      (Kuu + G / noise) alpha = b / noise,   m* = Kuu alpha*     (mu = Phi^T alpha, Kuu = kron_d K_d, K_d tridiagonal)
//     Markov:  (Kuu^-1 + G / noise) m = b / noise                         (mu = Psi^T m, Kuu^-1 = kron_d of tridiagonals)
// with G = sum_n w_n w_n^T and b = sum_n w_n y_n.  One pass over the binned observations assembles G and b: a lane sums its
// run in registers (observation dtype) and flushes once per run with float64 atomics.  Jacobi-preconditioned CG in float64
// solves the system; its scalars live in a device status record, so the host only reads that record between batches.
//
// G is stored symmetrically, (3^D + 1) / 2 coefficients per node, [slot][node]: with the stencil index
// k = sum_d (o_d + 1) 3^(D-1-d) of an offset o and the centre kc = (3^D - 1) / 2, slot k - kc of node i holds G[i][i + o] for
// k >= kc; G[i][i + o] with k < kc is slot 3^D - 1 - k - kc of node i + o.  The 3-D product reads 14 coefficients per node
// from memory instead of 27; the mirrored ones come from neighbouring nodes, which the same CTA or L2 has just read.
//
// The per-lane code (enter / observe / flush) is __host__ __device__ like bin_lane_* so that the SIMT emulator executes it.
#pragma once
#include "obs_binned.cuh"
#include "svgpm.cuh"

namespace vggp {

template <int D> struct MoSlots { static constexpr int v = (Pow3<D>::v + 1) / 2; };

// flush of one cell: b[corner] and the symmetric slots of G for every pair of corners i <= j whose nodes exist (`live` bit
// mask).  `pair(i, j, p)` gives sum w_i w_j of pair number p (pairs in the order of the two loops).
template <int D, typename Pair, typename Adder>
VGGP_HD void mo_flush_cell(const int (&stride)[D], int64_t M, int64_t base, unsigned live, const Pair& pair,
                           const double (&by)[1 << D], double* G, double* b, const Adder& add) {
    constexpr int NC = 1 << D, KC = (Pow3<D>::v - 1) / 2;
    int p = 0;
#pragma unroll
    for (int i = 0; i < NC; ++i) {
        int64_t oi = 0;
#pragma unroll
        for (int d = 0; d < D; ++d) oi += ((i >> (D - 1 - d)) & 1) ? stride[d] : 0;
        if ((live >> i) & 1u) add(b + base + oi, by[i]);
#pragma unroll
        for (int j = i; j < NC; ++j, ++p) {
            if (!((live >> i) & (live >> j) & 1u)) continue;
            // i < j: the first dimension where the corners differ has o_d = +1, so k > kc and node i owns the slot
            int k = 0;
#pragma unroll
            for (int d = 0; d < D; ++d) k = 3 * k + (((j >> (D - 1 - d)) & 1) - ((i >> (D - 1 - d)) & 1) + 1);
            add(G + (int64_t)(k - KC) * M + base + oi, pair(i, j, p));
        }
    }
}

// ---- B1: hat weights, sums as moments of a_d (as k_obs_b1_binned) ------------------------------------------------
template <typename T, int D>
struct MoB1Lane {
    int c[D];
    T tlo[D], h[D], rh[D];
    T gy[1 << D];                // sum y prod_{d in S} a_d, S indexed by bits (dimension 0 = most significant bit)
    T mom[Pow3<D>::v];           // sum prod_d a_d^{k_d}, index sum_d k_d 3^(D-1-d); entry 0 (the count) is not accumulated
};

template <typename T, int D>
VGGP_HD void mo_b1_enter(const BinGeom<D>& g, MoB1Lane<T, D>& s, uint32_t cell, const T* tab, const float* knots) {
    bin_decode_cell<D>(cell, g.K, s.c);
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const int n = g.K[d];
        const T* tb = tab + (g.tab_off[d] + s.c[d]);
        s.tlo[d] = (T)knots[g.knot_off[d] + s.c[d]];
        s.h[d] = tb[6 * n];
        s.rh[d] = tb[7 * n];
    }
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) s.gy[i] = (T)0;
#pragma unroll
    for (int i = 0; i < Pow3<D>::v; ++i) s.mom[i] = (T)0;
}

// padding slots (x = lower knot, so a_d = 0; y = 0) add nothing; `live` guards y all the same
template <typename T, int D>
VGGP_HD void mo_b1_obs(MoB1Lane<T, D>& s, const T (&x)[D], T y, bool live) {
    T w[D], w2[D];
#pragma unroll
    for (int d = 0; d < D; ++d) {
        w[d] = bin_div(x[d] - s.tlo[d], s.h[d], s.rh[d]);
        w2[d] = w[d] * w[d];
    }
    T mono[1 << D];
    mono[0] = (T)1;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const int bit = 1 << (D - 1 - d);
#pragma unroll
        for (int i = 0; i < (1 << D); ++i)
            if ((i & bit) && !(i & (bit - 1))) mono[i] = (i ^ bit) ? mono[i ^ bit] * w[d] : w[d];
    }
    const T yy = live ? y : (T)0;
    s.gy[0] += yy;
#pragma unroll
    for (int i = 1; i < (1 << D); ++i) s.gy[i] = bin_fma(yy, mono[i], s.gy[i]);
    // moments: products over dimensions 1..D-1 materialised, dimension 0 fused into the sums (as bin_lane_obs)
    constexpr int LEN = Pow3<D - 1>::v;
    T tp[LEN];
    tp[0] = (T)1;
    {
        int len = 1;
#pragma unroll
        for (int d = D - 1; d >= 1; --d) {
#pragma unroll
            for (int j = 0; j < LEN; ++j)
                if (j < len) {
                    tp[len + j] = (j == 0) ? w[d] : w[d] * tp[j];
                    tp[2 * len + j] = (j == 0) ? w2[d] : w2[d] * tp[j];
                }
            len *= 3;
        }
    }
#pragma unroll
    for (int j = 1; j < LEN; ++j) s.mom[j] += tp[j];
    s.mom[LEN] += w[0];
    s.mom[2 * LEN] += w2[0];
#pragma unroll
    for (int j = 1; j < LEN; ++j) {
        s.mom[LEN + j] = bin_fma(w[0], tp[j], s.mom[LEN + j]);
        s.mom[2 * LEN + j] = bin_fma(w2[0], tp[j], s.mom[2 * LEN + j]);
    }
}

// sum w_i w_j from the pair-type sums t[sum_d (bit_i + bit_j) 3^(D-1-d)] (type 0: (1-a)^2, 1: (1-a) a, 2: a^2)
template <int D>
struct MoTypePairs {
    const double* t;
    VGGP_HD double operator()(int i, int j, int) const {
        int k = 0;
#pragma unroll
        for (int d = 0; d < D; ++d) k = 3 * k + ((i >> (D - 1 - d)) & 1) + ((j >> (D - 1 - d)) & 1);
        return t[k];
    }
};

template <typename T, int D, typename Adder>
VGGP_HD void mo_b1_flush(const BinGeom<D>& g, int64_t M, const MoB1Lane<T, D>& s, int nrun, double* G, double* b,
                         const Adder& add) {
    constexpr int P3 = Pow3<D>::v;
    double t[P3];
#pragma unroll
    for (int i = 0; i < P3; ++i) t[i] = (double)s.mom[i];
    t[0] = (double)nrun;
    // per dimension (sum 1, sum a, sum a^2) -> (sum (1-a)^2, sum (1-a) a, sum a^2)
#pragma unroll
    for (int d = 0; d < D; ++d) {
        int st = 1;
#pragma unroll
        for (int e = d + 1; e < D; ++e) st *= 3;
#pragma unroll
        for (int i = 0; i < P3; ++i)
            if ((i / st) % 3 == 0) {
                const double m0 = t[i], m1 = t[i + st], m2 = t[i + 2 * st];
                t[i] = m0 - 2.0 * m1 + m2;
                t[i + st] = m1 - m2;
            }
    }
    // sums with y: monomial basis -> corner basis, per dimension (m0, m1) -> (m0 - m1, m1)
    double by[1 << D];
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) by[i] = (double)s.gy[i];
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const int bit = 1 << (D - 1 - d);
#pragma unroll
        for (int i = 0; i < (1 << D); ++i)
            if (!(i & bit)) by[i] -= by[i | bit];
    }
    int64_t base = 0;
#pragma unroll
    for (int d = 0; d < D; ++d) base += (int64_t)s.c[d] * g.stride[d];
    mo_flush_cell<D>(g.stride, M, base, (1u << (1 << D)) - 1u, MoTypePairs<D>{t}, by, G, b, add);
}

// ---- Markov: weights of svgpm_weights on the extended cells, corner products summed directly ---------------------
template <int D> struct MoPairs { static constexpr int v = (1 << D) * ((1 << D) + 1) / 2; };

template <typename T, int D>
struct MoSvmLane {
    int e[D];
    T c[D][SVM_TAB];
    bool vl[D], vr[D];
    T gg[MoPairs<D>::v];         // sum w_i w_j over corner pairs i <= j
    T gy[1 << D];                // sum w_i y
};

template <typename T, int D>
VGGP_HD void mo_svm_enter(const SvgpmGeom<D>& g, MoSvmLane<T, D>& s, uint32_t cell, const T* tab) {
    svgpm_decode_cell<D>(cell, g.M, s.e);
#pragma unroll
    for (int d = 0; d < D; ++d) {
        svgpm_load_cell<T, D>(g, tab, d, s.e[d], s.c[d]);
        s.vl[d] = s.e[d] == 0;
        s.vr[d] = s.e[d] == g.M[d];
    }
#pragma unroll
    for (int i = 0; i < MoPairs<D>::v; ++i) s.gg[i] = (T)0;
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) s.gy[i] = (T)0;
}

template <typename T, int D>
VGGP_HD void mo_svm_obs(MoSvmLane<T, D>& s, const T (&rl)[D], const T (&x)[D], T y, bool live) {
    if (!live) return;
    T w[D][2];
#pragma unroll
    for (int d = 0; d < D; ++d) {
        T u0, u1;
        svgpm_weights<T, false>(s.c[d], s.vl[d], s.vr[d], x[d], rl[d], w[d][0], w[d][1], u0, u1);
    }
    T wc[1 << D];
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) {
        T prod = (T)1;
#pragma unroll
        for (int d = 0; d < D; ++d) prod *= w[d][(i >> (D - 1 - d)) & 1];
        wc[i] = prod;
    }
    int p = 0;
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) {
        s.gy[i] = bin_fma(wc[i], y, s.gy[i]);
#pragma unroll
        for (int j = i; j < (1 << D); ++j, ++p) s.gg[p] = bin_fma(wc[i], wc[j], s.gg[p]);
    }
}

template <typename T>
struct MoListPairs {
    const T* v;
    VGGP_HD double operator()(int, int, int p) const { return (double)v[p]; }
};

// corners whose node does not exist (virtual cells outside the points) are dropped, as in svgpm_lane_flush
template <typename T, int D, typename Adder>
VGGP_HD void mo_svm_flush(const SvgpmGeom<D>& g, int64_t M, const MoSvmLane<T, D>& s, double* G, double* b,
                          const Adder& add) {
    unsigned live = 0;
    int64_t base = 0;
#pragma unroll
    for (int d = 0; d < D; ++d) base += (int64_t)(s.e[d] - 1) * g.stride[d];
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) {
        bool ok = true;
#pragma unroll
        for (int d = 0; d < D; ++d) ok = ok && svgpm_node<D>(g, d, s.e[d], (i >> (D - 1 - d)) & 1) >= 0;
        live |= ok ? (1u << i) : 0u;
    }
    double by[1 << D];
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) by[i] = (double)s.gy[i];
    mo_flush_cell<D>(g.stride, M, base, live, MoListPairs<T>{s.gg}, by, G, b, add);
}

}  // namespace vggp

// ---------------------------------------------------------------------------------------------------------
// Device side
// ---------------------------------------------------------------------------------------------------------
#if (defined(__CUDACC__) || defined(VGGP_EMUL)) && !defined(VGGP_HOST_EMUL)
namespace vggp {

// K1m (B1): one pass over the binned layout, same streaming as k_obs_b1_binned (persistent warps, longest task first,
// register ping-pong of the next group).  G ([MoSlots][M]) and b (M) zeroed before.
template <typename T, int D>
__global__ void __launch_bounds__(BIN_THREADS, (bin_min_blocks<T, D>()))
k_mo_b1_assemble(const __grid_constant__ BinnedArgs<T, D> a, double* __restrict__ G, double* __restrict__ b, i64 M) {
    const int lane = threadIdx.x & 31;
    const AtomicAdder add;
    BinLane<T, D> unused;
    MoB1Lane<T, D> s;
    BinTask<T, D> t;
    const T* tab = reinterpret_cast<const T*>(a.tables);
    const float* knots = reinterpret_cast<const float*>(a.tables + a.knots_byte_off);
    bool first = true;
    while (bin_next_task<T, D, false>(a, lane, unused, t, first)) {
        T xa[D][4], ya[4], xb[D][4], yb[4];
        bin_load_group<T, D>(t.base, xa, ya);
        mo_b1_enter<T, D>(a.geo, s, t.cell, tab, knots);
#pragma unroll 1
        for (int gi = 0; gi < t.groups; gi += 2) {
            if (gi + 1 < t.groups) bin_load_group<T, D>(t.base + (i64)(gi + 1) * ((D + 1) * 128), xb, yb);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                T xx[D];
#pragma unroll
                for (int d = 0; d < D; ++d) xx[d] = xa[d][j];
                mo_b1_obs<T, D>(s, xx, ya[j], 4 * gi + j < t.nrun);
            }
            if (gi + 2 < t.groups) bin_load_group<T, D>(t.base + (i64)(gi + 2) * ((D + 1) * 128), xa, ya);
            if (gi + 1 < t.groups) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    T xx[D];
#pragma unroll
                    for (int d = 0; d < D; ++d) xx[d] = xb[d][j];
                    mo_b1_obs<T, D>(s, xx, yb[j], 4 * (gi + 1) + j < t.nrun);
                }
            }
        }
        if (t.valid) mo_b1_flush<T, D>(a.geo, M, s, t.nrun, G, b, add);
    }
}

// K1m (Markov): the same streaming over extended cells (as k_obs_svgpm_binned); lengthscales of the last grid forward
template <typename T, int D>
__global__ void __launch_bounds__(BIN_THREADS)
k_mo_svm_assemble(const __grid_constant__ SvgpmArgs<T, D> a, double* __restrict__ G, double* __restrict__ b, i64 M) {
    const int lane = threadIdx.x & 31;
    const AtomicAdder add;
    T rl[D];
#pragma unroll
    for (int d = 0; d < D; ++d) rl[d] = (T)(1.0 / a.theta[d]);
    BinLane<T, D> unused;
    MoSvmLane<T, D> s;
    BinTask<T, D> t;
    bool first = true;
    while (bin_next_task<T, D, false>(a.bin, lane, unused, t, first)) {
        T xa[D][4], ya[4], xb[D][4], yb[4];
        bin_load_group<T, D>(t.base, xa, ya);
        mo_svm_enter<T, D>(a.geo, s, t.cell, a.tab);
#pragma unroll 1
        for (int gi = 0; gi < t.groups; gi += 2) {
            if (gi + 1 < t.groups) bin_load_group<T, D>(t.base + (i64)(gi + 1) * ((D + 1) * 128), xb, yb);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                T xx[D];
#pragma unroll
                for (int d = 0; d < D; ++d) xx[d] = xa[d][j];
                mo_svm_obs<T, D>(s, rl, xx, ya[j], 4 * gi + j < t.nrun);
            }
            if (gi + 2 < t.groups) bin_load_group<T, D>(t.base + (i64)(gi + 2) * ((D + 1) * 128), xa, ya);
            if (gi + 1 < t.groups) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    T xx[D];
#pragma unroll
                    for (int d = 0; d < D; ++d) xx[d] = xb[d][j];
                    mo_svm_obs<T, D>(s, rl, xx, yb[j], 4 * (gi + 1) + j < t.nrun);
                }
            }
        }
        if (t.valid) mo_svm_flush<T, D>(a.geo, M, s, G, b, add);
    }
}

// ---- grid side: Jacobi-preconditioned CG ----------------------------------------------------------------------
// Device status of a solve.  Kernels of iteration k: k_mo_matvec (rz <- rz_acc, clears the accumulators, pq += p.q),
// k_mo_update (x, r, rz_acc += r.z, rr_acc += r.r), k_mo_direction (p, clears pq, counts the iteration, sets `done` once
// ||r|| <= rtol ||rhs||).  Every field is written by one kernel and read by later ones only, so no launch needs a grid-wide
// barrier; once `done` is set every kernel returns at once.
struct MoStatus {
    double bb;                   // ||b / noise||^2
    double rz, pq, rz_acc, rr_acc, relres;
    int iters, done;
};

template <int D>
struct MoSys {
    i64 M;
    int n[D], stride[D];
    const double* bd[D];         // diagonal of the prior factor of dimension d (B1: K_d, Markov: K_d^-1)
    const double* bo[D];         // its first off diagonal, bo[i] = A_d[i][i + 1] (0 at i = n - 1)
    const double* G;             // [MoSlots][M]
    const double* theta;         // theta of the last grid forward (noise = theta[2 D])
};

// row u of (kron_d A_d + G / noise) x (WITH_G) or of kron_d A_d x; `diag`: the row's diagonal entry
template <int D, bool WITH_G, typename X>
__device__ __forceinline__ double mo_row(const MoSys<D>& s, i64 u, const X* __restrict__ x, double inv_noise, double* diag) {
    constexpr int P3 = Pow3<D>::v, KC = (P3 - 1) / 2;
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
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < P3; ++k) {
        int kk = k;
        i64 off = 0;
        bool ok = true;
        double cp = 1.0;
#pragma unroll
        for (int d = D - 1; d >= 0; --d) {
            const int o = kk % 3;
            kk /= 3;
            const int j = idx[d] + o - 1;
            ok = ok && j >= 0 && j < s.n[d];
            off += (i64)(o - 1) * s.stride[d];
            cp *= c[d][o];
        }
        if (!ok) continue;
        if (WITH_G) cp += inv_noise * (k >= KC ? s.G[(i64)(k - KC) * s.M + u] : s.G[(i64)(P3 - 1 - k - KC) * s.M + u + off]);
        acc = fma(cp, (double)x[u + off], acc);
    }
    if (diag) {
        double dg = 1.0;
#pragma unroll
        for (int d = 0; d < D; ++d) dg *= c[d][1];
        *diag = WITH_G ? dg + inv_noise * s.G[u] : dg;
    }
    return acc;
}

// B1 prior factor bands K_d (the entries k_build_factors uses), [bd | bo] per dimension.  grid (ceil(max M_d / 256), D)
__global__ void __launch_bounds__(256) k_mo_b1_bands(const __grid_constant__ GridDims g, const double* __restrict__ theta,
                                                     double* __restrict__ band, int band_stride) {
    const int d = blockIdx.y, n = g.n[d];
    const int i = (int)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double* bd = band + (i64)d * band_stride;
    bd[i] = factor_entry(g, theta, d, i, i);
    bd[n + i] = i + 1 < n ? factor_entry(g, theta, d, i, i + 1) : 0.0;
}

// x = x0, r = b / noise - A x0, dinv = 1 / diag(A), p = dinv r; ||b / noise||^2, r.z, r.r into the (zeroed) status
template <typename X, int D>
__global__ void __launch_bounds__(256) k_mo_init(const __grid_constant__ MoSys<D> s, const double* __restrict__ b,
                                                 const X* __restrict__ x0, double* __restrict__ x, double* __restrict__ r,
                                                 double* __restrict__ p, double* __restrict__ dinv, MoStatus* st) {
    __shared__ double red[32];
    const double inv_noise = 1.0 / s.theta[2 * D];
    double bb = 0.0, rz = 0.0, rr = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < s.M; u += (i64)gridDim.x * blockDim.x) {
        double dg;
        const double ax = mo_row<D, true, X>(s, u, x0, inv_noise, &dg);
        const double rhs = b[u] * inv_noise, ri = rhs - ax, di = 1.0 / dg;
        x[u] = (double)x0[u];
        r[u] = ri;
        p[u] = di * ri;
        dinv[u] = di;
        bb = fma(rhs, rhs, bb);
        rz = fma(ri * di, ri, rz);
        rr = fma(ri, ri, rr);
    }
    bb = block_sum(bb, red);
    rz = block_sum(rz, red);
    rr = block_sum(rr, red);
    if (threadIdx.x == 0) { atomicAdd(&st->bb, bb); atomicAdd(&st->rz_acc, rz); atomicAdd(&st->rr_acc, rr); }
}

template <int D>
__global__ void __launch_bounds__(256) k_mo_matvec(const __grid_constant__ MoSys<D> s, const double* __restrict__ p,
                                                   double* __restrict__ q, MoStatus* st) {
    __shared__ double red[32];
    if (st->done) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) { st->rz = st->rz_acc; st->rz_acc = 0.0; st->rr_acc = 0.0; }
    const double inv_noise = 1.0 / s.theta[2 * D];
    double pq = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < s.M; u += (i64)gridDim.x * blockDim.x) {
        const double v = mo_row<D, true, double>(s, u, p, inv_noise, nullptr);
        q[u] = v;
        pq = fma(p[u], v, pq);
    }
    pq = block_sum(pq, red);
    if (threadIdx.x == 0) atomicAdd(&st->pq, pq);
}

__global__ void __launch_bounds__(256) k_mo_update(i64 M, const double* __restrict__ p, const double* __restrict__ q,
                                                   const double* __restrict__ dinv, double* __restrict__ x,
                                                   double* __restrict__ r, MoStatus* st) {
    __shared__ double red[32];
    if (st->done) return;
    const double alpha = st->rz / st->pq;
    double rz = 0.0, rr = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < M; u += (i64)gridDim.x * blockDim.x) {
        x[u] = fma(alpha, p[u], x[u]);
        const double ri = fma(-alpha, q[u], r[u]);
        r[u] = ri;
        rz = fma(ri * dinv[u], ri, rz);
        rr = fma(ri, ri, rr);
    }
    rz = block_sum(rz, red);
    rr = block_sum(rr, red);
    if (threadIdx.x == 0) { atomicAdd(&st->rz_acc, rz); atomicAdd(&st->rr_acc, rr); }
}

// every block takes the same decision from the same status values; a converged solve leaves p as it is
__global__ void __launch_bounds__(256) k_mo_direction(i64 M, const double* __restrict__ r, const double* __restrict__ dinv,
                                                      double* __restrict__ p, double rtol, MoStatus* st) {
    if (st->done) return;
    const double relres = sqrt(st->rr_acc / st->bb);
    const bool conv = !(relres > rtol);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        st->pq = 0.0;
        st->iters += 1;
        st->relres = relres;
        if (conv) st->done = 1;
    }
    if (conv) return;
    const double beta = st->rz_acc / st->rz;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < M; u += (i64)gridDim.x * blockDim.x)
        p[u] = fma(beta, p[u], dinv[u] * r[u]);
}

// B1: m* = Kuu alpha*
template <int D>
__global__ void __launch_bounds__(256) k_mo_prior_apply(const __grid_constant__ MoSys<D> s, const double* __restrict__ x,
                                                        double* __restrict__ out) {
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < s.M; u += (i64)gridDim.x * blockDim.x)
        out[u] = mo_row<D, false, double>(s, u, x, 0.0, nullptr);
}

// ---- grid side: CG preconditioned by kron_d (F_d + g I)^-1 ---------------------------------------------------------
// F_d is the tridiagonal prior factor of dimension d (MoSys::bd / bo) and g = (sum_u G[u][u] / (noise M))^(1 / D), so
// kron_d (F_d + g I) matches the prior and the mean data diagonal of the system.  One application is D tridiagonal solves,
// one per mode of the row-major (M_1, ..., M_D) tensor.  Per dimension the Thomas factors [l | 1 / d' | off] (n each):
//     forward   y_i = x_i - l_i y_{i-1}                     (l_0 = 0)
//     backward  z_i = (y_i - off_i z_{i+1}) / d'_i          (off_{n-1} = 0)
// Kernels of one Kronecker iteration: k_mo_matvec, k_mo_kron_update (x, r, rr_acc), D x k_mo_kron_sweep (z = P r, the last
// one adds r.z to rz_acc), k_mo_kron_direction (p = z + beta p).  The Jacobi kernels above are not used by this solve.
struct MoKron {
    double gsum;                 // sum_u G[0][u], the trace of G
};
template <int D> struct MoFacOff { int off[D]; };      // offset of dimension d's factors: 3 sum_{e < d} M_e

// trace of G (slot 0 is the diagonal) into k->gsum (zeroed before)
__global__ void __launch_bounds__(256) k_mo_kron_trace(i64 M, const double* __restrict__ G, MoKron* k) {
    __shared__ double red[32];
    double acc = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < M; u += (i64)gridDim.x * blockDim.x) acc += G[u];
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) atomicAdd(&k->gsum, acc);
}

// Thomas LU of F_d + g I, one thread per dimension (SPD tridiagonal: no pivoting).  fac + fac_off[d]: [l | 1 / d' | off]
template <int D>
__global__ void __launch_bounds__(32) k_mo_kron_factors(const __grid_constant__ MoSys<D> s, const MoKron* k,
                                                        double* __restrict__ fac, const __grid_constant__ MoFacOff<D> fo) {
    const int d = threadIdx.x;
    if (d >= D) return;
    const double g = pow(fmax(k->gsum, 0.0) / (s.theta[2 * D] * (double)s.M), 1.0 / D);
    const int n = s.n[d];
    const double* bd = s.bd[d];
    const double* bo = s.bo[d];
    double* l = fac + fo.off[d];
    double* invd = l + n;
    double* off = invd + n;
    double dinv = 1.0 / (bd[0] + g);
    l[0] = 0.0;
    invd[0] = dinv;
    for (int i = 1; i < n; ++i) {
        const double o = bo[i - 1], li = o * dinv;
        dinv = 1.0 / (bd[i] + g - li * o);
        l[i] = li;
        invd[i] = dinv;
        off[i - 1] = o;
    }
    off[n - 1] = 0.0;
}

// Tridiagonal solve along one mode, in place or from `in` to `out`.  The mode has n nodes and stride `inner`; its F = M / n
// fibres are f = outer * inner + j at elements outer * n * inner + j + i * inner.  Each fibre is cut into S segments of Ls
// nodes, one thread per (fibre, segment), so short fibre counts still fill the GPU.  An affine map x -> a x + b composes in
// either order, so each segment needs only its own elements to know its start values:
//   1. (S > 1) compose the forward map of the segment from a zero start: one read;
//   2. chain the forward maps of the fibre's earlier segments in shared memory into this segment's start value y_{lo-1};
//      run the exact forward recurrence from it, writing y, and compose the backward map of the segment from the y it
//      produces: one read, one write;
//   3. chain the backward maps of the later segments into z_{hi}; run the exact backward recurrence: one read, one write.
//   STAGED = false (modes d < D - 1): thread t is fibre t % FB of segment t / FB, FB = 32 consecutive fibres per segment, so
//                  a warp reads 32 consecutive doubles at every step.  Global traffic per element: 3 reads and 2 writes
//                  (2 and 2 with S = 1); the second and third passes re-read what the block has just touched.
//   STAGED = true  (the contiguous mode, inner = 1): the block's FB rows are one contiguous range, copied into shared memory
//                  with coalesced loads, swept there, and written back the same way (one global read and one write per
//                  element); thread t is segment t % S of row t / S, and segment s of a row starts at s * P in shared
//                  memory with P = Ls | 1, so a half warp reads 16 different banks.
// RZ (STAGED only: the last sweep of an application is the contiguous mode): also add r.z over the block's elements into
// st->rz_acc.
struct MoSweep {
    i64 F, inner;
    int n, S, Ls, P;
    const double* fac;           // [l | 1 / d' | off] of this dimension
};

template <bool STAGED, bool RZ>
__global__ void __launch_bounds__(1024) k_mo_kron_sweep(const __grid_constant__ MoSweep w, const double* in, double* out,
                                                        const double* __restrict__ r, MoStatus* st) {
    static_assert(STAGED || !RZ, "r.z is accumulated by the staged sweep of the contiguous mode");
    __shared__ double sa[1024], sb[1024], red[32];
    extern __shared__ double sm[];
    if (st->done) return;
    const int tid = threadIdx.x, S = w.S, FB = (int)blockDim.x / S, n = w.n;
    const int seg = STAGED ? tid % S : tid / FB, fl = STAGED ? tid / S : tid % FB;
    const i64 f0 = (i64)blockIdx.x * FB, f = f0 + fl;
    const bool act = f < w.F;
    const int lo = min(n, seg * w.Ls), hi = min(n, lo + w.Ls);
    const double* __restrict__ l = w.fac;
    const double* __restrict__ invd = l + n;
    const double* __restrict__ off = invd + n;
    // element i of this thread's fibre: src[i * step], dst[i * step]
    const double* src;
    double* dst;
    i64 step;
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
    } else {
        const i64 outer = f / w.inner, j = f - outer * w.inner, base = outer * n * w.inner + j;
        src = in + base;
        dst = out + base;
        step = w.inner;
    }
    auto idx = [&](int s2) { return STAGED ? fl * S + s2 : s2 * FB + fl; };

    // 1. forward map of the segment, y_{hi-1} = A y_{lo-1} + B
    double A = 1.0, B = 0.0, c = 0.0;
    if (S > 1) {
        if (act)
            for (int i = lo; i < hi; ++i) { B = fma(-l[i], B, src[i * step]); A *= -l[i]; }
        sa[tid] = A; sb[tid] = B;
        __syncthreads();
        for (int s2 = 0; s2 < seg; ++s2) c = fma(sa[idx(s2)], c, sb[idx(s2)]);
        __syncthreads();
    }
    // 2. forward recurrence from y_{lo-1} = c; backward map z_lo = A z_hi + B composed along the way
    //    (z_i = a_i z_{i+1} + b_i with a_i = -off_i / d'_i, b_i = y_i / d'_i)
    A = 1.0; B = 0.0;
    if (act)
        for (int i = lo; i < hi; ++i) {
            c = fma(-l[i], c, src[i * step]);
            dst[i * step] = c;
            B = fma(A, c * invd[i], B);
            A *= -off[i] * invd[i];
        }
    // 3. backward recurrence from z_hi
    c = 0.0;
    if (S > 1) {
        sa[tid] = A; sb[tid] = B;
        __syncthreads();
        for (int s2 = S - 1; s2 > seg; --s2) c = fma(sa[idx(s2)], c, sb[idx(s2)]);
    }
    if (act)
        for (int i = hi - 1; i >= lo; --i) {
            c = fma(-off[i], c, dst[i * step]) * invd[i];
            dst[i * step] = c;
        }
    if (STAGED) {
        double rz = 0.0;
        __syncthreads();
        for (i64 j = tid; j < nrows * n; j += blockDim.x) {
            const int row = (int)(j / n), i = (int)(j - (i64)row * n);
            const double v = sm[(i64)row * S * w.P + (i / w.Ls) * w.P + i % w.Ls];
            out[f0 * n + j] = v;
            if (RZ) rz = fma(r[f0 * n + j], v, rz);
        }
        if (RZ) {
            rz = block_sum(rz, red);
            if (tid == 0) atomicAdd(&st->rz_acc, rz);
        }
    }
}

// x = x0, r = b / noise - A x0; ||b / noise||^2 and r.r into the (zeroed) status.  r.z comes from the first application.
template <typename X, int D>
__global__ void __launch_bounds__(256) k_mo_kron_init(const __grid_constant__ MoSys<D> s, const double* __restrict__ b,
                                                      const X* __restrict__ x0, double* __restrict__ x,
                                                      double* __restrict__ r, MoStatus* st) {
    __shared__ double red[32];
    const double inv_noise = 1.0 / s.theta[2 * D];
    double bb = 0.0, rr = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < s.M; u += (i64)gridDim.x * blockDim.x) {
        const double ax = mo_row<D, true, X>(s, u, x0, inv_noise, nullptr);
        const double rhs = b[u] * inv_noise, ri = rhs - ax;
        x[u] = (double)x0[u];
        r[u] = ri;
        bb = fma(rhs, rhs, bb);
        rr = fma(ri, ri, rr);
    }
    bb = block_sum(bb, red);
    rr = block_sum(rr, red);
    if (threadIdx.x == 0) { atomicAdd(&st->bb, bb); atomicAdd(&st->rr_acc, rr); }
}

__global__ void __launch_bounds__(256) k_mo_kron_update(i64 M, const double* __restrict__ p, const double* __restrict__ q,
                                                        double* __restrict__ x, double* __restrict__ r, MoStatus* st) {
    __shared__ double red[32];
    if (st->done) return;
    const double alpha = st->rz / st->pq;
    double rr = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < M; u += (i64)gridDim.x * blockDim.x) {
        x[u] = fma(alpha, p[u], x[u]);
        const double ri = fma(-alpha, q[u], r[u]);
        r[u] = ri;
        rr = fma(ri, ri, rr);
    }
    rr = block_sum(rr, red);
    if (threadIdx.x == 0) atomicAdd(&st->rr_acc, rr);
}

// as k_mo_direction with p = z + beta p
__global__ void __launch_bounds__(256) k_mo_kron_direction(i64 M, const double* __restrict__ z, double* __restrict__ p,
                                                           double rtol, MoStatus* st) {
    if (st->done) return;
    const double relres = sqrt(st->rr_acc / st->bb);
    const bool conv = !(relres > rtol);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        st->pq = 0.0;
        st->iters += 1;
        st->relres = relres;
        if (conv) st->done = 1;
    }
    if (conv) return;
    const double beta = st->rz_acc / st->rz;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < M; u += (i64)gridDim.x * blockDim.x)
        p[u] = fma(beta, p[u], z[u]);
}

}  // namespace vggp
#endif
