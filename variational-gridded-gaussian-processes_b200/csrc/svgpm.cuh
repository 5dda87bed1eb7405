// Product-grid SVGP in its O(1)-per-observation Markov form (family VGGP_SVGP_MARKOV, DESIGN.md section 4, K1f).
//
// K_d = s2_d exp(-|z_i - z_j| / l_d) on sorted points is the covariance of an Ornstein-Uhlenbeck process, so K_d^-1 is
// tridiagonal and psi_d(x) = K_d^-1 k_d(Z, x) has two non-zeros: with the extended cell e = #{z < x} in 0..M_d (e = 0 and
// e = M_d are virtual cells outside the points) and its nodes e - 1 (weight wlo) and e (weight whi),
//     in a cell of width h:  a = (z_e - x) / l,  b = (x - z_{e-1}) / l,  wlo = sinh(a) / sinh(h / l),  whi = sinh(b) / sinh(h / l)
//     left of z_0:  whi = exp(-a);   right of z_{M-1}:  wlo = exp(-b)
// and, in the unwhitened parametrisation,
//     mu = sum_corners prod_d w_d m[corner],   var = prod s2_d - prod_d w_d^T K_d[e] w_d + prod_d w_d^T S_d[e] w_d
// with K_d[e], S_d[e] the 2 x 2 diagonal blocks of K_d and S_d = tril(L_d) tril(L_d)^T (oracle/svgp_markov.py).
//
// Per-cell table of dimension d (observation dtype, [SVM_TAB][M_d + 1]): t0, t1 (the cell's knots), kx = s2 rho,
// slo, sx, shi (S block), u = 1 / (1 - rho^2), ceta = (h / l) (2 u - 1) = (h / l) coth(h / l).  Per-dimension float64 bands
// for the reverse pass ([SVM_W][M_d]): diag / off of K_d^-1 and their l-derivatives, kx and its l-derivative, S diag / off.
//
// The per-lane code (enter / observe / flush) is __host__ __device__ like bin_lane_* so that the SIMT emulator executes it.
#pragma once
#include "obs_binned.cuh"

namespace vggp {

enum { SVM_T0 = 0, SVM_T1, SVM_KX, SVM_SLO, SVM_SX, SVM_SHI, SVM_U, SVM_CETA, SVM_TAB };
enum { SVW_PD = 0, SVW_PO, SVW_DPD, SVW_DPO, SVW_KX, SVW_DKX, SVW_SD, SVW_SO, SVM_W };
// plan scalars of the family (float64): per dimension log det K_d, log det S_d, tr(K_d^-1 S_d), its l-derivative, the
// l-derivative of log det K_d (grid forward); m^T K^-1 m and its l-derivatives (grid backward)
enum { SVS_LDK = 0, SVS_LDS = 3, SVS_TR = 6, SVS_DTR = 9, SVS_DLDK = 12, SVS_MKM = 15, SVS_DMKM = 16, SVS_COUNT = 20 };

template <int D>
struct SvgpmGeom {
    int M[D];            // inducing points per dimension
    int stride[D];       // row-major strides of m
    int band_off[D];     // [bp_d | bp_o | bq_d | bq_o] of dimension d inside the band block, M_d values each
    int tab_off[D];      // dimension d inside the cell table ([SVM_TAB][M_d + 1])
};

VGGP_HD float svm_expm1(float v) { return expm1f(v); }
VGGP_HD double svm_expm1(double v) { return expm1(v); }

// weights of one dimension (and their l-derivatives with bands fixed if `dw`).  c: the cell's table row, e: extended cell.
template <typename T, bool DW>
VGGP_HD void svgpm_weights(const T (&c)[SVM_TAB], bool vl, bool vr, T x, T rl, T& wlo, T& whi, T& dlo, T& dhi) {
    T a = (c[SVM_T1] - x) * rl, b = (x - c[SVM_T0]) * rl;
    a = a > (T)0 ? a : (T)0;
    b = b > (T)0 ? b : (T)0;
    const T ema = svm_expm1(-a), emb = svm_expm1(-b);
    const T Ea = (T)1 + ema, Eb = (T)1 + emb, u = c[SVM_U];
    // 1 - exp(-2a) = -ema (2 + ema): exact for small a (l >> h), no overflow for large a
    T lo = Eb * (-ema * ((T)2 + ema)) * u, hi = Ea * (-emb * ((T)2 + emb)) * u;
    lo = vl ? (T)0 : (vr ? Eb : lo);
    hi = vr ? (T)0 : (vl ? Ea : hi);
    wlo = lo;
    whi = hi;
    if (DW) {
        // d sinh(a)/sinh(eta) / dl = (eta coth(eta) wlo - a cosh(a) / sinh(eta)) / l,  cosh(a) / sinh(eta) = Eb (1 + Ea^2) u
        T dl = (c[SVM_CETA] * lo - a * Eb * ((T)1 + Ea * Ea) * u) * rl;
        T dh = (c[SVM_CETA] * hi - b * Ea * ((T)1 + Eb * Eb) * u) * rl;
        dl = vl ? (T)0 : (vr ? lo * b * rl : dl);
        dh = vr ? (T)0 : (vl ? hi * a * rl : dh);
        dlo = dl;
        dhi = dh;
    }
}

template <typename T, int D>
struct SvgpmLane {
    int e[D];
    T c[D][SVM_TAB];
    bool vl[D], vr[D];
    T mc[1 << D];                // m at the cell's corners (0 where a node does not exist)
    T gm[1 << D];                // sum r prod_d w_d
    T bp[D][3], bq[D][3];        // sum prod_{e != d} p_e (wlo^2, wlo whi, whi^2)_d, the same with q
    T gl[D];                     // sum d/dl_d [(y - mu)^2 + var], bands fixed
    T acc;                       // sum r^2 - prod p + prod q
};

template <int D>
VGGP_HD void svgpm_decode_cell(uint32_t cell, const int (&M)[D], int (&e)[D]) {
#pragma unroll
    for (int d = D - 1; d >= 0; --d) {
        const uint32_t E = (uint32_t)(M[d] + 1);
        e[d] = (int)(cell % E);
        cell /= E;
    }
}

// node index of slot `hi` (0: e - 1, 1: e) of dimension d, or -1
template <int D>
VGGP_HD int svgpm_node(const SvgpmGeom<D>& g, int d, int e, int hi) {
    const int i = e - 1 + hi;
    return (i >= 0 && i < g.M[d]) ? i : -1;
}

template <typename T, int D>
VGGP_HD void svgpm_load_cell(const SvgpmGeom<D>& g, const T* tab, int d, int e, T (&c)[SVM_TAB]) {
    const int E = g.M[d] + 1;
#pragma unroll
    for (int k = 0; k < SVM_TAB; ++k) c[k] = tab[g.tab_off[d] + k * E + e];
}

// corner values of m for the cells e[0..D-1]
template <typename T, int D>
VGGP_HD void svgpm_corners(const SvgpmGeom<D>& g, const int (&e)[D], const T* m, T (&mc)[1 << D]) {
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) {
        int off = 0;
        bool ok = true;
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const int nd = svgpm_node<D>(g, d, e[d], (i >> (D - 1 - d)) & 1);
            ok = ok && nd >= 0;
            off += (nd >= 0 ? nd : 0) * g.stride[d];
        }
        mc[i] = ok ? bin_ldg(m + off) : (T)0;
    }
}

template <typename T, int D>
VGGP_HD void svgpm_lane_enter(const SvgpmGeom<D>& g, SvgpmLane<T, D>& s, uint32_t cell, const T* tab, const T* m) {
    svgpm_decode_cell<D>(cell, g.M, s.e);
#pragma unroll
    for (int d = 0; d < D; ++d) {
        svgpm_load_cell<T, D>(g, tab, d, s.e[d], s.c[d]);
        s.vl[d] = s.e[d] == 0;
        s.vr[d] = s.e[d] == g.M[d];
#pragma unroll
        for (int k = 0; k < 3; ++k) { s.bp[d][k] = (T)0; s.bq[d][k] = (T)0; }
        s.gl[d] = (T)0;
    }
    svgpm_corners<T, D>(g, s.e, m, s.mc);
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) s.gm[i] = (T)0;
    s.acc = (T)0;
}

// p_d = w^T K_d[e] w (diagonal s2), q_d = w^T S_d[e] w and the half gradients K w, S w
template <typename T>
VGGP_HD void svgpm_forms(const T (&c)[SVM_TAB], T s2, T wlo, T whi, T& p, T& q, T (&kw)[2], T (&sw)[2]) {
    kw[0] = s2 * wlo + c[SVM_KX] * whi;
    kw[1] = c[SVM_KX] * wlo + s2 * whi;
    sw[0] = c[SVM_SLO] * wlo + c[SVM_SX] * whi;
    sw[1] = c[SVM_SX] * wlo + c[SVM_SHI] * whi;
    p = wlo * kw[0] + whi * kw[1];
    q = wlo * sw[0] + whi * sw[1];
}

// one observation of the run; padding slots (`live` false) contribute nothing
template <typename T, int D>
VGGP_HD void svgpm_lane_obs(SvgpmLane<T, D>& s, const T (&s2)[D], const T (&rl)[D], const T (&x)[D], T y, bool live) {
    if (!live) return;
    T w[D][2], dw[D][2], p[D], q[D], kw[D][2], sw[D][2];
#pragma unroll
    for (int d = 0; d < D; ++d) {
        svgpm_weights<T, true>(s.c[d], s.vl[d], s.vr[d], x[d], rl[d], w[d][0], w[d][1], dw[d][0], dw[d][1]);
        svgpm_forms<T>(s.c[d], s2[d], w[d][0], w[d][1], p[d], q[d], kw[d], sw[d]);
    }
    T mu = (T)0, dmu[D];
#pragma unroll
    for (int d = 0; d < D; ++d) dmu[d] = (T)0;
    T wc[1 << D];
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) {
        T prod = (T)1;
#pragma unroll
        for (int d = 0; d < D; ++d) prod *= w[d][(i >> (D - 1 - d)) & 1];
        wc[i] = prod;
        mu = bin_fma(prod, s.mc[i], mu);
#pragma unroll
        for (int d = 0; d < D; ++d) {
            T o = s.mc[i] * dw[d][(i >> (D - 1 - d)) & 1];
#pragma unroll
            for (int f = 0; f < D; ++f)
                if (f != d) o *= w[f][(i >> (D - 1 - f)) & 1];
            dmu[d] += o;
        }
    }
    const T r = y - mu;
    T pp = p[0], qq = q[0];
#pragma unroll
    for (int d = 1; d < D; ++d) { pp *= p[d]; qq *= q[d]; }
    s.acc += bin_fma(r, r, qq - pp);
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) s.gm[i] = bin_fma(r, wc[i], s.gm[i]);
#pragma unroll
    for (int d = 0; d < D; ++d) {
        T op = (T)1, oq = (T)1;
#pragma unroll
        for (int f = 0; f < D; ++f)
            if (f != d) { op *= p[f]; oq *= q[f]; }
        const T ll = w[d][0] * w[d][0], lh = w[d][0] * w[d][1], hh = w[d][1] * w[d][1];
        s.bp[d][0] = bin_fma(op, ll, s.bp[d][0]);
        s.bp[d][1] = bin_fma(op, lh, s.bp[d][1]);
        s.bp[d][2] = bin_fma(op, hh, s.bp[d][2]);
        s.bq[d][0] = bin_fma(oq, ll, s.bq[d][0]);
        s.bq[d][1] = bin_fma(oq, lh, s.bq[d][1]);
        s.bq[d][2] = bin_fma(oq, hh, s.bq[d][2]);
        const T dK = kw[d][0] * dw[d][0] + kw[d][1] * dw[d][1];
        const T dS = sw[d][0] * dw[d][0] + sw[d][1] * dw[d][1];
        s.gl[d] += (T)2 * (oq * dS - op * dK - r * dmu[d]);
    }
}

// leave the cell: corner sums into d m, band sums into the band block (nodes that exist only); returns the run's
// sum r^2 - prod p + prod q and adds its lengthscale sums to gl_out
template <typename T, int D, typename Adder>
VGGP_HD T svgpm_lane_flush(const SvgpmGeom<D>& g, const SvgpmLane<T, D>& s, T* gm_out, T* gband, double (&gl_out)[D],
                           const Adder& add) {
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) {
        int off = 0;
        bool ok = true;
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const int nd = svgpm_node<D>(g, d, s.e[d], (i >> (D - 1 - d)) & 1);
            ok = ok && nd >= 0;
            off += (nd >= 0 ? nd : 0) * g.stride[d];
        }
        if (ok) add(gm_out + off, s.gm[i]);
    }
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const int n = g.M[d];
        const int lo = svgpm_node<D>(g, d, s.e[d], 0), hi = svgpm_node<D>(g, d, s.e[d], 1);
        T* b = gband + g.band_off[d];
        if (lo >= 0) { add(b + lo, s.bp[d][0]); add(b + 2 * n + lo, s.bq[d][0]); }
        if (hi >= 0) { add(b + hi, s.bp[d][2]); add(b + 2 * n + hi, s.bq[d][2]); }
        if (lo >= 0 && hi >= 0) { add(b + n + lo, s.bp[d][1]); add(b + 3 * n + lo, s.bq[d][1]); }
        gl_out[d] += (double)s.gl[d];
    }
    return s.acc;
}

// mean and variance at one point (prediction)
template <typename T, int D>
VGGP_HD void svgpm_point(const SvgpmGeom<D>& g, const T* tab, const T* m, const T (&s2)[D], const T (&rl)[D],
                         const int (&e)[D], const T (&x)[D], T& mu, T& var) {
    T w[D][2], p[D], q[D], kff = (T)1;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        T c[SVM_TAB], kw[2], sw[2], dummy0, dummy1;
        svgpm_load_cell<T, D>(g, tab, d, e[d], c);
        svgpm_weights<T, false>(c, e[d] == 0, e[d] == g.M[d], x[d], rl[d], w[d][0], w[d][1], dummy0, dummy1);
        svgpm_forms<T>(c, s2[d], w[d][0], w[d][1], p[d], q[d], kw, sw);
        kff *= s2[d];
    }
    T mc[1 << D];
    svgpm_corners<T, D>(g, e, m, mc);
    mu = (T)0;
#pragma unroll
    for (int i = 0; i < (1 << D); ++i) {
        T prod = (T)1;
#pragma unroll
        for (int d = 0; d < D; ++d) prod *= w[d][(i >> (D - 1 - d)) & 1];
        mu = bin_fma(prod, mc[i], mu);
    }
    T pp = p[0], qq = q[0];
#pragma unroll
    for (int d = 1; d < D; ++d) { pp *= p[d]; qq *= q[d]; }
    var = kff - pp + qq;
}

}  // namespace vggp

// ---------------------------------------------------------------------------------------------------------
// Device side
// ---------------------------------------------------------------------------------------------------------
#if (defined(__CUDACC__) || defined(VGGP_EMUL)) && !defined(VGGP_HOST_EMUL)
namespace vggp {

template <typename T, int D>
struct SvgpmArgs {
    BinnedArgs<T, D> bin;            // task / run streaming, band replicas, gbuf scalars (obs_binned.cuh)
    SvgpmGeom<D> geo;
    const T* tab;                    // per-cell tables
    const T* m;                      // m in the observation dtype
    const double* theta;             // theta of the last grid forward (device)
};

// K1f: fused per-observation forward + backward over the binned layout with extended cells (k_b0s_keys / k_b0s_gather)
template <typename T, int D>
__global__ void __launch_bounds__(BIN_THREADS) k_obs_svgpm_binned(const __grid_constant__ SvgpmArgs<T, D> a) {
    __shared__ double red[32];
    const int lane = threadIdx.x & 31;
    const AtomicAdder add;
    T s2[D], rl[D];
#pragma unroll
    for (int d = 0; d < D; ++d) { s2[d] = (T)a.theta[D + d]; rl[d] = (T)(1.0 / a.theta[d]); }
    double etot = 0.0, gl[D];
#pragma unroll
    for (int d = 0; d < D; ++d) gl[d] = 0.0;
    BinLane<T, D> unused;
    SvgpmLane<T, D> s;
    BinTask<T, D> t;
    T* const gband = a.bin.gband + (i64)(blockIdx.x % (unsigned)a.bin.n_rep) * a.bin.band_rep_stride;
    bool first = true;
    while (bin_next_task<T, D, false>(a.bin, lane, unused, t, first)) {
        T xa[D][4], ya[4], xb[D][4], yb[4];
        bin_load_group<T, D>(t.base, xa, ya);
        svgpm_lane_enter<T, D>(a.geo, s, t.cell, a.tab, a.m);
#pragma unroll 1
        for (int gi = 0; gi < t.groups; gi += 2) {
            if (gi + 1 < t.groups) bin_load_group<T, D>(t.base + (i64)(gi + 1) * ((D + 1) * 128), xb, yb);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                T xx[D];
#pragma unroll
                for (int d = 0; d < D; ++d) xx[d] = xa[d][j];
                svgpm_lane_obs<T, D>(s, s2, rl, xx, ya[j], 4 * gi + j < t.nrun);
            }
            if (gi + 2 < t.groups) bin_load_group<T, D>(t.base + (i64)(gi + 2) * ((D + 1) * 128), xa, ya);
            if (gi + 1 < t.groups) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    T xx[D];
#pragma unroll
                    for (int d = 0; d < D; ++d) xx[d] = xb[d][j];
                    svgpm_lane_obs<T, D>(s, s2, rl, xx, yb[j], 4 * (gi + 1) + j < t.nrun);
                }
            }
        }
        if (t.valid) etot += (double)svgpm_lane_flush<T, D>(a.geo, s, a.bin.galpha, gband, gl, add);
    }
    bin_finish<T, D>(a.bin, etot, red);
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const double v = block_sum(gl[d], red);
        if (threadIdx.x == 0) atomicAdd(a.bin.gs + 3 + d, v);
    }
}

// ---- grid forward ---------------------------------------------------------------------------------------
struct SvgpmGrid {
    int D, M[3];
    const float* z[3];               // knots = inducing locations
    i64 Loff[3];
    double* W[3];                    // [SVM_W][M_d] float64 bands
    void* tab;                       // per-cell tables (observation dtype)
    int tab_off[3];
    double* sc;                      // SVS_COUNT scalars
    int* info;
};

// one warp per node row i of dimension blockIdx.y: S_d band by row dot products of tril(L_d), the closed-form K_d^-1 band,
// its log det and the trace, the cell table.  grid (ceil(max M_d / 8), D), 256 threads; sc[0 .. SVS_MKM) and info zeroed before.
template <typename T>
__global__ void __launch_bounds__(256) k_svgpm_fwd(const __grid_constant__ SvgpmGrid g, const double* __restrict__ theta,
                                                   const double* __restrict__ L) {
    const int d = blockIdx.y, n = g.M[d], D = g.D;
    const int i = (int)blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    const double* Ld = L + g.Loff[d];
    const double* Li = Ld + (i64)i * n;
    const double* Lj = Li + n;                      // row i + 1
    double sii = 0.0, sio = 0.0, sjj = 0.0;
    for (int k = lane; k <= i; k += 32) {
        sii = fma(Li[k], Li[k], sii);
        if (i + 1 < n) sio = fma(Li[k], Lj[k], sio);
    }
    if (i + 1 < n)
        for (int k = lane; k <= i + 1; k += 32) sjj = fma(Lj[k], Lj[k], sjj);
    sii = warp_sum(sii);
    sio = warp_sum(sio);
    sjj = warp_sum(sjj);
    if (lane != 0) return;
    const double l = theta[d], s2 = theta[D + d], rl = 1.0 / l;
    auto hgt = [&](int c) { return (double)g.z[d][c + 1] - (double)g.z[d][c]; };
    // u_c = 1 / (1 - rho_c^2) with expm1 (l >> h is the normal regime), du / dl = u (u - 1) 2 h / l^2
    auto ucell = [&](int c) { return -1.0 / expm1(-2.0 * hgt(c) * rl); };
    double pd, dpd;
    {
        double uu = 0.0, du = 0.0;
        if (i > 0) { const double u = ucell(i - 1); uu += u; du += u * (u - 1.0) * 2.0 * hgt(i - 1) * rl * rl; }
        if (i + 1 < n) { const double u = ucell(i); uu += u; du += u * (u - 1.0) * 2.0 * hgt(i) * rl * rl; }
        if (i > 0 && i + 1 < n) uu -= 1.0;
        pd = uu / s2;
        dpd = du / s2;
    }
    double* W = g.W[d];
    W[SVW_PD * n + i] = pd;
    W[SVW_DPD * n + i] = dpd;
    W[SVW_SD * n + i] = sii;
    double tr = pd * sii, dtr = dpd * sii, ldk = (i == 0) ? (double)n * log(s2) : 0.0, dldk = 0.0;
    T* tab = reinterpret_cast<T*>(g.tab) + g.tab_off[d];
    const int E = n + 1;
    if (i + 1 < n) {
        const double h = hgt(i), eta = h * rl, rho = exp(-eta), u = ucell(i);
        const double po = -rho * u / s2, dpo = -rho * u * h * rl * rl * (2.0 * u - 1.0) / s2;
        W[SVW_PO * n + i] = po;
        W[SVW_DPO * n + i] = dpo;
        W[SVW_KX * n + i] = s2 * rho;
        W[SVW_DKX * n + i] = s2 * rho * h * rl * rl;
        W[SVW_SO * n + i] = sio;
        tr += 2.0 * po * sio;
        dtr += 2.0 * dpo * sio;
        ldk -= log(u);
        dldk -= (u - 1.0) * 2.0 * h * rl * rl;
        const int e = i + 1;
        tab[SVM_T0 * E + e] = (T)g.z[d][i];
        tab[SVM_T1 * E + e] = (T)g.z[d][i + 1];
        tab[SVM_KX * E + e] = (T)(s2 * rho);
        tab[SVM_SLO * E + e] = (T)sii;
        tab[SVM_SX * E + e] = (T)sio;
        tab[SVM_SHI * E + e] = (T)sjj;
        tab[SVM_U * E + e] = (T)u;
        tab[SVM_CETA * E + e] = (T)(eta * (2.0 * u - 1.0));
    } else {
        W[SVW_PO * n + i] = 0.0; W[SVW_DPO * n + i] = 0.0; W[SVW_KX * n + i] = 0.0; W[SVW_DKX * n + i] = 0.0;
        W[SVW_SO * n + i] = 0.0;
    }
    // virtual cells: e = 0 (left of z_0, node 0 only) and e = M (right of z_{M-1}, node M - 1 only)
    if (i == 0 || i + 1 == n) {
        const int e = (i == 0) ? 0 : n;
        tab[SVM_T0 * E + e] = (T)g.z[d][i];
        tab[SVM_T1 * E + e] = (T)g.z[d][i];
        tab[SVM_KX * E + e] = (T)0;
        tab[SVM_SLO * E + e] = (T)(e == 0 ? 0.0 : sii);
        tab[SVM_SX * E + e] = (T)0;
        tab[SVM_SHI * E + e] = (T)(e == 0 ? sii : 0.0);
        tab[SVM_U * E + e] = (T)1;
        tab[SVM_CETA * E + e] = (T)0;
    }
    const double Lii = Li[i];
    atomicAdd(g.sc + SVS_LDK + d, ldk);
    atomicAdd(g.sc + SVS_LDS + d, 2.0 * log(fabs(Lii)));
    atomicAdd(g.sc + SVS_TR + d, tr);
    atomicAdd(g.sc + SVS_DTR + d, dtr);
    atomicAdd(g.sc + SVS_DLDK + d, dldk);
    if (Lii == 0.0 || !(l > 0.0) || !(s2 > 0.0) || !isfinite(l) || !isfinite(s2) || !isfinite(Lii)) atomicMax(g.info, d + 1);
}

// ---- grid backward --------------------------------------------------------------------------------------
struct SvgpmBwd {
    int D, M[3], stride[3], band_off[3];
    i64 Mtot, Loff[3];
    const double* W[3];
    double* sc;
};

// dm = (ell_scale / noise) g_m - (kron_d K_d^-1) m as one 3^D-point stencil, with the reductions m^T K^-1 m and
// m^T (dK_d^-1/dl_d x_{e != d} K_e^-1) m.  grid-stride, 256 threads; sc[SVS_MKM ..] zeroed before.
template <typename T, int D>
__global__ void __launch_bounds__(256) k_svgpm_dm(const __grid_constant__ SvgpmBwd g, const T* __restrict__ gm,
                                                  const double* __restrict__ m, const double* __restrict__ theta,
                                                  double ell_scale, double* __restrict__ dm) {
    __shared__ double red[32];
    const double cg = ell_scale / theta[2 * D];
    double amk = 0.0, adk[D];
#pragma unroll
    for (int d = 0; d < D; ++d) adk[d] = 0.0;
    for (i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x; u < g.Mtot; u += (i64)gridDim.x * blockDim.x) {
        int idx[D];
        i64 rem = u;
#pragma unroll
        for (int d = 0; d < D; ++d) { idx[d] = (int)(rem / g.stride[d]); rem -= (i64)idx[d] * g.stride[d]; }
        double coef[D][3], dcoef[D][3];
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const int n = g.M[d], i = idx[d];
            const double* W = g.W[d];
            coef[d][1] = W[SVW_PD * n + i];
            dcoef[d][1] = W[SVW_DPD * n + i];
            coef[d][0] = i > 0 ? W[SVW_PO * n + i - 1] : 0.0;
            dcoef[d][0] = i > 0 ? W[SVW_DPO * n + i - 1] : 0.0;
            coef[d][2] = i + 1 < n ? W[SVW_PO * n + i] : 0.0;
            dcoef[d][2] = i + 1 < n ? W[SVW_DPO * n + i] : 0.0;
        }
        double km = 0.0, dkm[D];
#pragma unroll
        for (int d = 0; d < D; ++d) dkm[d] = 0.0;
        constexpr int NB3 = D == 1 ? 3 : (D == 2 ? 9 : 27);
        for (int k = 0; k < NB3; ++k) {
            int kk = k, off = 0;
            bool ok = true;
            int o[D];
#pragma unroll
            for (int d = D - 1; d >= 0; --d) {
                o[d] = kk % 3;
                kk /= 3;
                const int j = idx[d] + o[d] - 1;
                ok = ok && j >= 0 && j < g.M[d];
                off += (o[d] - 1) * g.stride[d];
            }
            if (!ok) continue;
            const double mj = m[u + off];
            double c = 1.0;
#pragma unroll
            for (int d = 0; d < D; ++d) c *= coef[d][o[d]];
            km = fma(c, mj, km);
#pragma unroll
            for (int d = 0; d < D; ++d) {
                double cd = dcoef[d][o[d]];
#pragma unroll
                for (int f = 0; f < D; ++f)
                    if (f != d) cd *= coef[f][o[f]];
                dkm[d] = fma(cd, mj, dkm[d]);
            }
        }
        dm[u] = cg * (double)gm[u] - km;
        amk = fma(m[u], km, amk);
#pragma unroll
        for (int d = 0; d < D; ++d) adk[d] = fma(m[u], dkm[d], adk[d]);
    }
    const double v = block_sum(amk, red);
    if (threadIdx.x == 0) atomicAdd(g.sc + SVS_MKM, v);
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const double w = block_sum(adk[d], red);
        if (threadIdx.x == 0) atomicAdd(g.sc + SVS_DMKM + d, w);
    }
}

// dL_d = tril( 2 cQ G_d L_d - c_d K_d^-1 L_d + (M / M_d) diag(1 / L_ii) ),  G_d = banded sums of the S band (gbuf),
// cQ = -ell_scale / (2 noise), c_d = prod_{e != d} tr(K_e^-1 S_e).  grid (ceil(max M_d^2 / 256), D)
template <typename T>
__global__ void __launch_bounds__(256) k_svgpm_dL(const __grid_constant__ SvgpmBwd g, const T* __restrict__ gband,
                                                  const double* __restrict__ L, const double* __restrict__ theta,
                                                  double ell_scale, double* __restrict__ dL) {
    const int d = blockIdx.y, n = g.M[d], D = g.D;
    const i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (i64)n * n) return;
    const int i = (int)(e / n), j = (int)(e % n);
    double v = 0.0;
    if (j <= i) {
        const double* Ld = L + g.Loff[d];
        const double* W = g.W[d];
        const T* b = gband + g.band_off[d];
        const double Lij = Ld[e];
        const double Lm = (i > 0 && j <= i - 1) ? Ld[e - n] : 0.0;        // tril(L)[i-1][j]
        const double Lp = (i + 1 < n) ? Ld[e + n] : 0.0;                  // tril(L)[i+1][j] (j <= i < i+1)
        const double gq = (double)b[2 * n + i] * Lij + (i > 0 ? (double)b[3 * n + i - 1] * Lm : 0.0)
                          + (i + 1 < n ? (double)b[3 * n + i] * Lp : 0.0);
        const double kl = W[SVW_PD * n + i] * Lij + (i > 0 ? W[SVW_PO * n + i - 1] * Lm : 0.0) + W[SVW_PO * n + i] * Lp;
        double c = 1.0;
        for (int f = 0; f < D; ++f)
            if (f != d) c *= g.sc[SVS_TR + f];
        v = -(ell_scale / theta[2 * D]) * gq - c * kl;
        if (i == j) v += ((double)g.Mtot / (double)n) / Lij;
    }
    dL[g.Loff[d] + e] = v;
}

// d theta and the ELBO.  One CTA of 256 threads.
template <typename T>
__global__ void __launch_bounds__(256) k_svgpm_theta(const __grid_constant__ SvgpmBwd g, const T* __restrict__ gband,
                                                     const double* __restrict__ gs,
                                                     const double* __restrict__ theta, double ell_scale,
                                                     double* __restrict__ out, double* __restrict__ dtheta) {
    __shared__ double red[32];
    const int D = g.D;
    double pp = 0.0, bl[3] = {0.0, 0.0, 0.0};
    for (int d = 0; d < D; ++d) {
        const int n = g.M[d];
        const double* W = g.W[d];
        const T* b = gband + g.band_off[d];
        const double s2 = theta[D + d];
        double a = 0.0, c = 0.0;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            if (d == 0) a += s2 * (double)b[i] + 2.0 * W[SVW_KX * n + i] * (double)b[n + i];
            c += 2.0 * W[SVW_DKX * n + i] * (double)b[n + i];
        }
        if (d == 0) pp = block_sum(a, red);
        bl[d] = block_sum(c, red);
    }
    if (threadIdx.x != 0) return;
    const double noise = theta[2 * D], E = gs[0], N = gs[1], Md = (double)g.Mtot;
    double kff = 1.0, trp = 1.0, lds = 0.0;
    for (int d = 0; d < D; ++d) {
        kff *= theta[D + d];
        trp *= g.sc[SVS_TR + d];
        lds += (Md / (double)g.M[d]) * (g.sc[SVS_LDK + d] - g.sc[SVS_LDS + d]);
    }
    const double mkm = g.sc[SVS_MKM];
    const double tot = E + N * kff;
    const double ell = -0.5 * N * log(2.0 * 3.14159265358979323846 * noise) - tot / (2.0 * noise);
    const double kl = 0.5 * (trp + mkm - Md + lds);
    out[0] = ell_scale * ell - kl;
    out[1] = ell_scale * ell;
    out[2] = kl;
    out[3] = N;
    for (int d = 0; d < D; ++d) {
        const double s2 = theta[D + d];
        double c = 1.0;
        for (int f = 0; f < D; ++f)
            if (f != d) c *= g.sc[SVS_TR + f];
        dtheta[d] = -ell_scale / (2.0 * noise) * (gs[3 + d] - bl[d])
                    - 0.5 * (c * g.sc[SVS_DTR + d] + g.sc[SVS_DMKM + d] + (Md / (double)g.M[d]) * g.sc[SVS_DLDK + d]);
        dtheta[D + d] = -ell_scale * (N * kff - pp) / (2.0 * noise * s2) + 0.5 * (trp + mkm - Md) / s2;
    }
    dtheta[2 * D] = ell_scale * (-N / (2.0 * noise) + tot / (2.0 * noise * noise));
}

// ---- prediction -------------------------------------------------------------------------------------------
template <typename T, int D>
struct SvgpmPredictArgs {
    SvgpmGeom<D> geo;
    const float* z[D];
    const T* x[D];
    const T* y;                      // metrics only
    i64 n;
    const T* tab;
    const T* m;
    const double* theta;
    T* mean;
    T* var;
    double* out;                     // metrics: { sum (t - p)^2, sum |t - p|, sum (t - t0), sum (t - t0)^2 }
};

template <typename T, int D, bool METRICS>
__global__ void __launch_bounds__(256) k_predict_svgpm(const __grid_constant__ SvgpmPredictArgs<T, D> a) {
    __shared__ double red[32];
    T s2[D], rl[D];
#pragma unroll
    for (int d = 0; d < D; ++d) { s2[d] = (T)a.theta[D + d]; rl[d] = (T)(1.0 / a.theta[d]); }
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    const double t0 = METRICS ? (double)a.y[0] : 0.0;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (i64)gridDim.x * blockDim.x) {
        int e[D];
        T x[D];
#pragma unroll
        for (int d = 0; d < D; ++d) {
            x[d] = a.x[d][i];
            e[d] = lower_bound_knots<T>(a.z[d], a.geo.M[d], x[d]);
        }
        T mu, var;
        svgpm_point<T, D>(a.geo, a.tab, a.m, s2, rl, e, x, mu, var);
        if (METRICS) {
            const double t = (double)a.y[i], r = t - (double)mu;
            acc[0] += r * r; acc[1] += fabs(r); acc[2] += t - t0; acc[3] += (t - t0) * (t - t0);
        } else {
            a.mean[i] = mu;
            a.var[i] = var;
        }
    }
    if (METRICS) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double v = block_sum(acc[k], red);
            if (threadIdx.x == 0) atomicAdd(a.out + k, v);
        }
    }
}

}  // namespace vggp
#endif
